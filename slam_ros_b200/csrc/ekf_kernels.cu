/* ekf_kernels.cu -- hand-written sm_100a kernels of libekfcuda (single filter, optionally row-sharded).
 *
 * Arithmetic contract: every expression that feeds the association gate, the gain or the covariance
 * follows the scalar expansion of the GSL reference-BLAS loop the reference calls at the cited line of
 * slam_ros/Robot.cpp (SURVEY.md appendix A): same operand order, same accumulation order, one rounding
 * per operation.  The explicit __dmul_rn/__dadd_rn/__dsub_rn intrinsics are never contracted into FMAs
 * (the file is also compiled with -fmad=false).  What differs from the reference by design: only the
 * UPPER triangle of P is kept (the reference's full-matrix update lets P drift asymmetric by ulps),
 * and sin/cos are CUDA's (<= 2 ulp) instead of glibc's.
 */
#include "ekf_internal.h"
#include "ekf_device.cuh"
#include <stdlib.h>
#include <string.h>
#include <cuda.h>
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

#define EKF_BLOCK 256

namespace {

__device__ __forceinline__ int owner_of_row(const EkfGeom& g, int r) { return (r / EKF_TILE) % g.world; }
__device__ __forceinline__ size_t local_row(const EkfGeom& g, int r) {
  return (size_t)((r / EKF_TILE) / g.world) * EKF_TILE + (size_t)(r % EKF_TILE);
}
/* is (r,q), r <= q, one of the eagerly maintained elements? */
__device__ __forceinline__ bool is_hot(int r, int q) {
  return r <= 2 || q == r || (q == r + 1 && (r & 1));
}
/* hot element (r <= q) straight from its replica */
__device__ __forceinline__ double hot_value(const EkfGeom& g, const EkfBuffers& b, int r, int q) {
  if (r <= 2) return b.top[(size_t)r * g.ld + q];
  const int j = (r - 3) >> 1;
  if (r & 1) return b.diag[4 * j + (q - r)];   /* r = a: (a,a) or (a,b) */
  return b.diag[4 * j + 2];                    /* r = b: (b,b) */
}
/* current value of a COLD upper element (r < q) owned by this rank: base minus the pending terms in order */
__device__ __forceinline__ double cold_value(const EkfGeom& g, const EkfBuffers& b, int r, int q, int np) {
  double p = b.P[local_row(g, r) * g.ld + q];
  for (int i = 0; i < np; ++i)
    p = sub_rank2(p, b.KSp[(size_t)i * g.ld + r], b.Kp[(size_t)i * g.ld + q]);
  return p;
}
/* 3x3 robot block with the lower half mirrored from the authoritative upper half */
__device__ __forceinline__ void load_rr(const EkfGeom& g, const double* top, double A[3][3]) {
  for (int i = 0; i < 3; ++i)
    for (int k = i; k < 3; ++k) { const double v = top[(size_t)i * g.ld + k]; A[i][k] = v; A[k][i] = v; }
}

/* Robot.cpp:367-489 for one (line, landmark j) pair; reads only replicated hot data */
__device__ void eval_gate(const EkfGeom& g, const EkfBuffers& b, const double x_pre[3], int j,
                          double z0, double z1, const double R[4], Gate& G) {
  const int a = 3 + 2 * j, bb = a + 1;
  double Cm[5][5];                                                    /* P at rows/cols {0,1,2,a,b} */
  for (int i = 0; i < 3; ++i) {
    for (int k = i; k < 3; ++k) { const double v = b.top[(size_t)i * g.ld + k]; Cm[i][k] = v; Cm[k][i] = v; }
    const double va = b.top[(size_t)i * g.ld + a], vb = b.top[(size_t)i * g.ld + bb];
    Cm[i][3] = va; Cm[3][i] = va; Cm[i][4] = vb; Cm[4][i] = vb;
  }
  Cm[3][3] = b.diag[4 * j]; Cm[3][4] = b.diag[4 * j + 1]; Cm[4][3] = Cm[3][4]; Cm[4][4] = b.diag[4 * j + 2];
  gate_from_block(Cm, b.y[a], b.y[bb], x_pre, z0, z1, R, G);
}

/* ------------------------------------------------------------------------------------------------ */
/* Robot::Robot (Robot.cpp:20-35): P[0,0] = P[1,1] = 0.05; everything else was zero-filled by memset */
__global__ void k_init(EkfGeom g, EkfBuffers b) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    b.top[0] = 0.05;
    b.top[(size_t)g.ld + 1] = 0.05;
    b.top[(size_t)2 * g.ld + 2] = 0.0;
  }
}

/* Robot.cpp:130-258 (structured: SURVEY appendix A.2).  Also opens the scan: per-line tables. */
/* Robot.cpp:130-258 (+ the per-scan resets of :294) for thread gid of stride: the body of k_predict, also run as the
 * prologue of the one-barrier line loop (k_scan_lines2 with u != NULL: one launch less on the latency path of small maps).
 * carry != NULL: the scan continues a sweep group (DESIGN section 5) whose earlier scans left *carry pending terms; its own
 * terms are appended after them (pbase = -*carry), so the group's one sweep folds them all in order. */
__device__ __forceinline__ void predict_body(const EkfGeom& g, const EkfBuffers& b, const double* __restrict__ u,
                                             const double* __restrict__ x_t0, int m, int gid, int stride,
                                             const int* __restrict__ carry) {
  EkfDevState* st = b.st;
  const double* x = x_t0 ? x_t0 : st->pose;
  const double x0 = x[0], x1 = x[1], x2 = x[2];
  const double u0 = u[0], u2 = u[2];
  const double ang = add_rn(x2, __ddiv_rn(u2, 2.0));
  double ca, sa;
  cos_sin(ang, ca, sa);
  const double F02 = mul_rn(-u0, sa), F12 = mul_rn(u0, ca);               /* :157, :160 */
  const int nl = 3 + 2 * st->L;
  double* t0p = b.top; double* t1p = b.top + g.ld; const double* t2p = b.top + 2 * (size_t)g.ld;
  /* :242 rows 0,1 of Fx*P (== cols 0,1 of (.)Fx'): P[0,q] += F02 P[2,q], P[1,q] += F12 P[2,q] over the live columns, as a
   * coalesced sweep of 16-byte column pairs (the rows start on 2 KB boundaries; column 3 is the one unpaired entry) */
  if (gid < 2 && nl > 3) {                                            /* the two unpaired ends: columns 3 and nl - 1 */
    const int q = gid ? nl - 1 : 3;
    const double p2 = t2p[q];
    double a0 = add_rn(0.0, t0p[q]); axpy_skip(a0, F02, p2);
    double a1 = add_rn(0.0, t1p[q]); axpy_skip(a1, F12, p2);
    t0p[q] = a0; t1p[q] = a1;
  }
  for (int q = 4 + 2 * gid; q + 1 < nl - 1; q += 2 * stride) {        /* aligned pairs (4,5) .. (nl-3, nl-2) */
    const double2 p2 = *reinterpret_cast<const double2*>(t2p + q);
    double2 r0 = *reinterpret_cast<const double2*>(t0p + q), r1 = *reinterpret_cast<const double2*>(t1p + q);
    r0.x = add_rn(0.0, r0.x); axpy_skip(r0.x, F02, p2.x); r0.y = add_rn(0.0, r0.y); axpy_skip(r0.y, F02, p2.y);
    r1.x = add_rn(0.0, r1.x); axpy_skip(r1.x, F12, p2.x); r1.y = add_rn(0.0, r1.y); axpy_skip(r1.y, F12, p2.y);
    *reinterpret_cast<double2*>(t0p + q) = r0; *reinterpret_cast<double2*>(t1p + q) = r1;
  }
  for (int i = gid; i < m; i += stride) { b.jbest[i] = EKF_NO_MATCH; b.jsing[i] = EKF_NO_MATCH; b.jout[i] = -1; }
  if (gid == 0) {
    double A[3][3], T[3][3], Pn[3][3];
    load_rr(g, b.top, A);
    for (int j = 0; j < 3; ++j) {                                     /* :242 */
      double r0 = 0.0, r1 = 0.0, r2 = 0.0;
      axpy_skip(r0, 1.0, A[0][j]); axpy_skip(r1, 1.0, A[1][j]);
      axpy_skip(r0, F02, A[2][j]); axpy_skip(r1, F12, A[2][j]); axpy_skip(r2, 1.0, A[2][j]);
      T[0][j] = r0; T[1][j] = r1; T[2][j] = r2;
    }
    for (int i = 0; i < 3; ++i) {                                     /* :246 */
      double c0 = 0.0; c0 = add_rn(c0, mul_rn(T[i][0], 1.0)); c0 = add_rn(c0, mul_rn(T[i][2], F02));
      double c1 = 0.0; c1 = add_rn(c1, mul_rn(T[i][1], 1.0)); c1 = add_rn(c1, mul_rn(T[i][2], F12));
      Pn[i][0] = add_rn(0.0, c0); Pn[i][1] = add_rn(0.0, c1); Pn[i][2] = T[i][2];
    }
    const double Fu[3][3] = {{ca, 0.0, __ddiv_rn(mul_rn(-u0, sa), 2.0)},   /* :180-188 */
                             {sa, 1.0, __ddiv_rn(mul_rn(u0, ca), 2.0)},
                             {0.0, 0.0, 1.0}};
    const double qf = add_rn(__ddiv_rn(-1.0, add_rn(1.0, fabs(u0))), 1.0);   /* :215-218 */
    const double Q[3] = {mul_rn(g.enc_noise, qf), mul_rn(mul_rn(2.0, g.enc_noise), qf), mul_rn(g.enc_noise, qf)};
    double FQ[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    for (int k = 0; k < 3; ++k)                                       /* :250 (NN, Q diagonal) */
      for (int i = 0; i < 3; ++i) {
        const double t = mul_rn(1.0, Fu[i][k]);
        if (t != 0.0)
          for (int j = 0; j < 3; ++j) FQ[i][j] = add_rn(FQ[i][j], mul_rn(t, (j == k) ? Q[k] : 0.0));
      }
    for (int i = 0; i < 3; ++i)                                       /* :254, :258 */
      for (int j = i; j < 3; ++j) {
        double t = 0.0;
        for (int k = 0; k < 3; ++k) t = add_rn(t, mul_rn(FQ[i][k], Fu[j][k]));
        b.top[(size_t)i * g.ld + j] = add_rn(Pn[i][j], add_rn(0.0, mul_rn(1.0, t)));
      }
    st->x_pre[0] = add_rn(x0, mul_rn(u0, ca));                            /* :148 */
    st->x_pre[1] = add_rn(x1, mul_rn(u0, sa));
    st->x_pre[2] = add_rn(x2, u2);
    if (x_t0) { st->pose[0] = x0; st->pose[1] = x1; st->pose[2] = x2; }
    st->epoch += 1;                                                   /* matchSavedIndexes.clear(), :294 */
    st->pbase = carry ? -*carry : 0; st->np = 0;
    b.pidx[0] = 0; b.eidx[0] = 0;
  }
}
__global__ void __launch_bounds__(EKF_BLOCK) k_predict(EkfGeom g, EkfBuffers b, const double* __restrict__ u,
                                                       const double* __restrict__ x_t0, int m, const int* __restrict__ carry) {
  predict_body(g, b, u, x_t0, m, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x, carry);
}

/* Robot.cpp:313-501 for one line: every un-matched landmark is gated in parallel; first fit = the
 * lowest passing index (warp-shuffle min, then one atomicMin per block). */
__global__ void __launch_bounds__(EKF_BLOCK) k_associate(EkfGeom g, EkfBuffers b, const double* __restrict__ z,
                                                         const double* __restrict__ R, int line) {
  __shared__ int s_min[EKF_BLOCK / 32];
  const EkfDevState* st = b.st;
  const int L = st->L;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  int cand = EKF_NO_MATCH;
  if (j < L && b.matched[j] != st->epoch) {
    const double xp[3] = {st->x_pre[0], st->x_pre[1], st->x_pre[2]};
    const double Rl[4] = {R[4 * line], R[4 * line + 1], R[4 * line + 2], R[4 * line + 3]};
    Gate G;
    eval_gate(g, b, xp, j, z[2 * line], z[2 * line + 1], Rl, G);
    if (G.singular) atomicMin(&b.jsing[line], j);                   /* reported by k_end_scan_a if below the winner */
    else if (!gate_rejects_d2(G.d2, g.gate_d2max)) cand = j;          /* :489 */
  }
  cand = __reduce_min_sync(0xffffffffu, cand);
  if ((threadIdx.x & 31) == 0) s_min[threadIdx.x >> 5] = cand;
  __syncthreads();
  if (threadIdx.x < 32) {
    int v = (threadIdx.x < EKF_BLOCK / 32) ? s_min[threadIdx.x] : EKF_NO_MATCH;
    v = __reduce_min_sync(0xffffffffu, v);
    if (threadIdx.x == 0 && v != EKF_NO_MATCH) atomicMin(&b.jbest[line], v);
  }
}

/* Robot.cpp:516-560: gain rows for the matched landmark.
 * mode 0: K, KS from local data;  mode 1: only publish the cold H-column slices this rank owns into
 * colA/colB (zero elsewhere);  mode 2: K, KS from colA/colB (after the exchange);  mode 3: only the
 * winner's innovation / S into the state block. */
__global__ void __launch_bounds__(EKF_BLOCK) k_gain(EkfGeom g, EkfBuffers b, const double* __restrict__ z,
                                                    const double* __restrict__ R, int line, int j_override,
                                                    int mode, int max_batch) {
  __shared__ Gate sG;
  const EkfDevState* st = b.st;
  const int j = (j_override >= 0) ? j_override : b.jbest[line];
  if (j == EKF_NO_MATCH) return;
  const int np = b.pidx[line] - st->pbase;
  if (np >= max_batch) return;                    /* host flushes before this can happen */
  const int nl = 3 + 2 * st->L;
  const int a = 3 + 2 * j, bb = a + 1;
  if (threadIdx.x == 0 && mode != 1) {
    const double xp[3] = {st->x_pre[0], st->x_pre[1], st->x_pre[2]};
    const double Rl[4] = {R[4 * line], R[4 * line + 1], R[4 * line + 2], R[4 * line + 3]};
    eval_gate(g, b, xp, j, z[2 * line], z[2 * line + 1], Rl, sG);
    if (blockIdx.x == 0) {
      b.st->v[0] = sG.v[0]; b.st->v[1] = sG.v[1];
      for (int t = 0; t < 4; ++t) b.st->S[t] = sG.S[t];
    }
  }
  if (mode == 3) return;                          /* innovation tap only (ekf_associate) */
  __syncthreads();
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  const int stride = gridDim.x * blockDim.x;
  for (int r = gid; r < nl; r += stride) {
    /* current P[r,a], P[r,b] through the symmetric upper storage */
    double pa, pb;
    const int lo_a = min(r, a), hi_a = max(r, a), lo_b = min(r, bb), hi_b = max(r, bb);
    const bool hot_a = is_hot(lo_a, hi_a), hot_b = is_hot(lo_b, hi_b);
    if (mode == 2) {
      pa = hot_a ? hot_value(g, b, lo_a, hi_a) : b.colA[r];
      pb = hot_b ? hot_value(g, b, lo_b, hi_b) : b.colB[r];
    } else {
      const bool own_a = (g.world == 1) || owner_of_row(g, lo_a) == g.rank;
      const bool own_b = (g.world == 1) || owner_of_row(g, lo_b) == g.rank;
      pa = hot_a ? hot_value(g, b, lo_a, hi_a) : (own_a ? cold_value(g, b, lo_a, hi_a, np) : 0.0);
      pb = hot_b ? hot_value(g, b, lo_b, hi_b) : (own_b ? cold_value(g, b, lo_b, hi_b, np) : 0.0);
      if (mode == 1) {
        b.colA[r] = hot_a ? 0.0 : pa;
        b.colB[r] = hot_b ? 0.0 : pb;
        continue;
      }
    }
    /* P[r,0], P[r,1], P[r,2] */
    double p0, p1, p2;
    if (r <= 2) {
      p0 = b.top[(size_t)min(r, 0) * g.ld + max(r, 0)];
      p1 = b.top[(size_t)min(r, 1) * g.ld + max(r, 1)];
      p2 = b.top[(size_t)min(r, 2) * g.ld + max(r, 2)];
    } else {
      p0 = b.top[r]; p1 = b.top[(size_t)g.ld + r]; p2 = b.top[(size_t)2 * g.ld + r];
    }
    double2 Kr, KSr;
    gain_row(sG, p0, p1, p2, pa, pb, Kr, KSr);
    b.Kp[(size_t)np * g.ld + r] = Kr;
    b.KSp[(size_t)np * g.ld + r] = KSr;
  }
}

/* Robot.cpp:564-602 restricted to the hot elements (rows 0-2, 2x2 diagonal blocks) and the state
 * vector; the cold part of P -= KS K' is deferred to k_sweep.  Also the per-line bookkeeping
 * (:501-504, :309/:325/:493). */
__global__ void __launch_bounds__(EKF_BLOCK) k_apply(EkfGeom g, EkfBuffers b, int line, int j_override) {
  EkfDevState* st = b.st;
  const int j = (j_override >= 0) ? j_override : (j_override == -2 ? EKF_NO_MATCH : b.jbest[line]);
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  const int nm = b.pidx[line];
  const int np = nm - st->pbase;
  if (j == EKF_NO_MATCH) {
    if (gid == 0) {
      const int e = b.eidx[line];
      b.ext[e] = line;
      b.eidx[line + 1] = e + 1; b.pidx[line + 1] = nm; b.jout[line] = -1;
    }
    return;
  }
  const int stride = gridDim.x * blockDim.x;
  const int nl = 3 + 2 * st->L;
  const double2* K = b.Kp + (size_t)np * g.ld;
  const double2* KS = b.KSp + (size_t)np * g.ld;
  const double v0 = st->v[0], v1 = st->v[1];
  const double2 ks0 = KS[0], ks1 = KS[1], ks2 = KS[2];
  for (int q = 3 + gid; q < nl; q += stride) {
    const double2 kq = K[q];
    b.top[q] = sub_rank2(b.top[q], ks0, kq);                        /* :564-568 rows 0..2 */
    b.top[(size_t)g.ld + q] = sub_rank2(b.top[(size_t)g.ld + q], ks1, kq);
    b.top[(size_t)2 * g.ld + q] = sub_rank2(b.top[(size_t)2 * g.ld + q], ks2, kq);
    const double2 ksq = KS[q];
    const int jj = (q - 3) >> 1;
    if (q & 1) {                                                      /* q = a: (a,a), (a,b) */
      b.diag[4 * jj] = sub_rank2(b.diag[4 * jj], ksq, kq);
      b.diag[4 * jj + 1] = sub_rank2(b.diag[4 * jj + 1], ksq, K[q + 1]);
    } else {                                                          /* q = b: (b,b) */
      b.diag[4 * jj + 2] = sub_rank2(b.diag[4 * jj + 2], ksq, kq);
    }
    double t = 0.0;                                                   /* :585-589  y += K * delta */
    axpy_skip(t, kq.x, v0); axpy_skip(t, kq.y, v1);
    b.y[q] = add_rn(b.y[q], t);
  }
  if (gid == 0) {
    const double2 kk[3] = {K[0], K[1], K[2]};
    const double2 ks[3] = {ks0, ks1, ks2};
    for (int r = 0; r < 3; ++r)
      for (int q = r; q < 3; ++q)
        b.top[(size_t)r * g.ld + q] = sub_rank2(b.top[(size_t)r * g.ld + q], ks[r], kk[q]);
    double yn[3];
    for (int r = 0; r < 3; ++r) {                                     /* :579-589 */
      double t = 0.0;
      axpy_skip(t, kk[r].x, v0); axpy_skip(t, kk[r].y, v1);
      yn[r] = add_rn(st->x_pre[r], t);
    }
    normalize_radian(yn[2]);                                          /* :596-602 */
    for (int r = 0; r < 3; ++r) { b.y[r] = yn[r]; st->pose[r] = yn[r]; st->x_pre[r] = yn[r]; }
    b.matched[j] = st->epoch;                                         /* :501 */
    b.jout[line] = j;
    b.pidx[line + 1] = nm + 1; b.eidx[line + 1] = b.eidx[line];
    st->np = np + 1;                                                  /* read only by the next sweep */
  }
}

/* ------------------------------------------------------------------------------------------------ */
/* All observed lines of a scan in ONE launch (single-GPU path): a thread-block cluster walks the lines
 * in order; within a line the three phases (gate every landmark + first-fit, gain rows, hot updates +
 * bookkeeping) are separated by hardware cluster barriers instead of kernel boundaries.  The phases are
 * the bodies of k_associate / k_gain(mode 0) / k_apply; the winner's gate record travels through
 * b.gates so it is evaluated once, as in the reference (Robot.cpp:367-489 feeds :516-602). */
#define FL_MAXP 128                   /* most pending terms a line can see: the previous scan's (<= 64) + this scan's (<= 64) */
#define GATE_REC 24                   /* doubles per landmark in b.gates: the gate (14), P[0..2, a], P[0..2, b] (6) */

__device__ __forceinline__ void gate_store(double* rec, const Gate& G) {
  rec[0] = G.c; rec[1] = G.s; rec[2] = G.g;
  for (int t = 0; t < 4; ++t) { rec[3 + t] = G.S[t]; rec[7 + t] = G.Si[t]; }
  rec[11] = G.v[0]; rec[12] = G.v[1]; rec[13] = G.d2;
}
__device__ __forceinline__ void gate_load(const double* rec, Gate& G) {
  G.c = rec[0]; G.s = rec[1]; G.g = rec[2];
  for (int t = 0; t < 4; ++t) { G.S[t] = rec[3 + t]; G.Si[t] = rec[7 + t]; }
  G.v[0] = rec[11]; G.v[1] = rec[12]; G.d2 = rec[13]; G.singular = 0;
}

/* Hot update of the robot block (3x3 of P, pose) for one pending term: Robot.cpp:564-568 on rows/cols 0..2
 * and :579-602.  Every thread of the line-loop kernel keeps its own identical copy in registers. */
__device__ __forceinline__ void update_robot_block(const double2 kk[3], const double2 ks[3], double v0, double v1,
                                                   double A[3][3], double xp[3]) {
  for (int r = 0; r < 3; ++r)
    for (int q = r; q < 3; ++q) { A[r][q] = sub_rank2(A[r][q], ks[r], kk[q]); A[q][r] = A[r][q]; }
  double yn[3];
  for (int r = 0; r < 3; ++r) {
    double t = 0.0;
    axpy_skip(t, kk[r].x, v0); axpy_skip(t, kk[r].y, v1);
    yn[r] = add_rn(xp[r], t);
  }
  normalize_radian(yn[2]);
  xp[0] = yn[0]; xp[1] = yn[1]; xp[2] = yn[2];
}

/* one row of the gain phase: everything that has to come from memory, issued as independent loads.
 * The pending list seen by a line is [previous scan's terms whose sweep may still be in flight] followed by
 * [this scan's terms]; s_slot[i] is the slot of the i-th pending term, npt their number. */
struct GainRow {
  double p0, p1, p2, pa, pb;
  double2 v[8];          /* first chunk of the row's pending terms (K S row entries or K column entries) */
  int kind;              /* 0: hot (no corrections), 1: column part (r < a), 2: row part (r > b) */
};
struct PendingList {     /* i-th pending term lives in slot prev_slot0 + i (i < prev_cnt) or own_slot0 + i - prev_cnt */
  int prev_cnt, prev_slot0, own_slot0;
  __device__ __forceinline__ int slot(int i) const { return (i < prev_cnt) ? prev_slot0 + i : own_slot0 + (i - prev_cnt); }
};
__device__ __forceinline__ void gain_row_load(const EkfGeom& g, const EkfBuffers& b, const double A[3][3], int r, int j,
                                              int npt, const PendingList& pl, GainRow& d) {
  const int a = 3 + 2 * j, bb = a + 1;
  d.kind = 0;
  if (r <= 2) {
    d.p0 = A[r][0]; d.p1 = A[r][1]; d.p2 = A[r][2];
    d.pa = b.top[(size_t)r * g.ld + a]; d.pb = b.top[(size_t)r * g.ld + bb];
    return;
  }
  d.p0 = b.top[r]; d.p1 = b.top[(size_t)g.ld + r]; d.p2 = b.top[(size_t)2 * g.ld + r];
  if (r == a) { d.pa = b.diag[4 * j]; d.pb = b.diag[4 * j + 1]; }
  else if (r == bb) { d.pa = b.diag[4 * j + 1]; d.pb = b.diag[4 * j + 2]; }
  else if (r < a) {                                                   /* column parts: P[r,a], P[r,b] */
    const double* Pr = b.P + local_row(g, r) * g.ld;
    d.pa = Pr[a]; d.pb = Pr[bb];
    d.kind = 1;
#pragma unroll
    for (int t = 0; t < 8; ++t) if (t < npt) d.v[t] = b.KSp[(size_t)pl.slot(t) * g.ld + r];
  } else {                                                            /* row parts: P[a,r], P[b,r] */
    d.pa = b.P[local_row(g, a) * g.ld + r]; d.pb = b.P[local_row(g, bb) * g.ld + r];
    d.kind = 2;
#pragma unroll
    for (int t = 0; t < 8; ++t) if (t < npt) d.v[t] = b.Kp[(size_t)pl.slot(t) * g.ld + r];
  }
}
/* applies the pending terms to the two cold entries of row r (d.pa, d.pb) */
__device__ __forceinline__ void gain_row_correct(const EkfGeom& g, const EkfBuffers& b, int r, int npt, GainRow& d,
                                                 const PendingList& pl, const double2* s_ka, const double2* s_kb,
                                                 const double2* s_ksa, const double2* s_ksb) {
  if (d.kind == 1) {
    for (int i0 = 0; i0 < npt; i0 += 8) {
      if (i0 > 0) {
#pragma unroll
        for (int t = 0; t < 8; ++t) if (i0 + t < npt) d.v[t] = b.KSp[(size_t)pl.slot(i0 + t) * g.ld + r];
      }
#pragma unroll
      for (int t = 0; t < 8; ++t) if (i0 + t < npt) {
        d.pa = sub_rank2(d.pa, d.v[t], s_ka[i0 + t]);
        d.pb = sub_rank2(d.pb, d.v[t], s_kb[i0 + t]);
      }
    }
  } else if (d.kind == 2) {
    for (int i0 = 0; i0 < npt; i0 += 8) {
      if (i0 > 0) {
#pragma unroll
        for (int t = 0; t < 8; ++t) if (i0 + t < npt) d.v[t] = b.Kp[(size_t)pl.slot(i0 + t) * g.ld + r];
      }
#pragma unroll
      for (int t = 0; t < 8; ++t) if (i0 + t < npt) {
        d.pa = sub_rank2(d.pa, s_ksa[i0 + t], d.v[t]);
        d.pb = sub_rank2(d.pb, s_ksb[i0 + t], d.v[t]);
      }
    }
  }
}
__device__ __forceinline__ void gain_row_emit(const EkfGeom& g, const EkfBuffers& b, const Gate& G, int r, int out_slot,
                                              const GainRow& d) {
  double2 Kr, KSr;
  gain_row(G, d.p0, d.p1, d.p2, d.pa, d.pb, Kr, KSr);
  b.Kp[(size_t)out_slot * g.ld + r] = Kr;
  b.KSp[(size_t)out_slot * g.ld + r] = KSr;
}

/* ---- row-sharded mode: the H-column slices are exchanged INSIDE the line-loop kernel over NVLink peer memory.
 * Every rank owns an exchange buffer [2 parities][colA | colB][ld] doubles followed by 8 arrival flags; peers map
 * it (CUDA IPC) and store the slice entries they own straight into it, then publish an epoch in the flag word.
 * No NCCL call, no kernel boundary: one NVLink round trip per matched line. ---- */
__device__ __forceinline__ double* xchg_col(const EkfPeers& pe, const EkfGeom& g, int p, int par, int which) {
  return pe.xchg[p] + ((size_t)(2 * par + which)) * g.ld;
}
__device__ __forceinline__ unsigned long long* xchg_flags(const EkfPeers& pe, const EkfGeom& g, int p) {
  return reinterpret_cast<unsigned long long*>(pe.xchg[p] + (size_t)4 * g.ld);
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
/* called by ONE thread after a local barrier: tell every peer this rank's slice entries are in place, then wait
 * for theirs.  Bounded spin: a missing peer raises a sticky error instead of hanging the GPU. */
__device__ __forceinline__ void st_relaxed_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void xgpu_exchange_barrier(const EkfPeers& pe, const EkfGeom& g, unsigned long long epoch, int* sticky) {
  /* ONE system-scope fence orders every slice store of this GPU (made visible to this thread by the grid barrier)
   * before the flag stores, which can then be relaxed: a release store per peer would pay the fence 8 times */
  __threadfence_system();
  for (int p = 0; p < pe.world; ++p) st_relaxed_sys(xchg_flags(pe, g, p) + pe.rank, epoch);
  const unsigned long long* mine = xchg_flags(pe, g, pe.rank);
  for (int q = 0; q < pe.world; ++q) {
    long long spins = 0;
    while (ld_acquire_sys(mine + q) < epoch) {
      if (++spins > 40000000LL) { atomicOr(sticky, EKF_STICKY_XCHG); break; }
    }
  }
}

#ifdef EKF_LINE_TIMING
__device__ unsigned long long g_line_ts[64 * 16];
__device__ __forceinline__ unsigned long long gtimer() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define TS(slot) do { if (gtid == 0 && line - line0 < 64) g_line_ts[(line - line0) * 16 + (slot)] = gtimer(); } while (0)
#else
#define TS(slot) do { } while (0)
#endif

/* Dependency chain per line: [landmark data + previous K] -> gate -> atomicMin -> barrier -> [winner]
 * -> [gate record + row data] -> gain -> barrier: three memory round trips and two cluster barriers. */
/* The 256-thread form is capped at 85 registers (3 CTAs/SM bound): measured on B200, a CTA of it is then
 * co-scheduled next to a resident sweep CTA (105 regs x 288 threads, 148 KB); at 118+ registers it is not. */
/* COOP = false: the CTAs form one thread-block cluster and synchronise with the hardware cluster barrier.
 * COOP = true : the same CTAs are launched cooperatively and synchronise with a grid barrier instead, so
 *               they need not sit in one GPC -- this is the form that runs on the SMs the overlapped sweep
 *               leaves free (see enqueue_scan_overlapped). */
template <int FL_THREADS, bool COOP, bool SHARD>
__global__ void __launch_bounds__(FL_THREADS, FL_THREADS == 256 ? 3 : 1) k_scan_lines(EkfGeom g, EkfBuffers b, const double* __restrict__ z,
                                                              const double* __restrict__ R, int line0, int line1,
                                                              int own_slot0, int prev_slot0, const int* __restrict__ prev_cnt_ptr,
                                                              EkfPeers pe) {
  __shared__ int s_min[FL_THREADS / 32];
  __shared__ double2 s_ka[FL_MAXP], s_kb[FL_MAXP], s_ksa[FL_MAXP], s_ksb[FL_MAXP];
  const int prev_cnt = prev_cnt_ptr ? *prev_cnt_ptr : 0;   /* previous scan's terms not yet folded into b.P */
  EkfDevState* st = b.st;
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x;      /* the grid is exactly one cluster / one co-resident group */
  const int gstride = gridDim.x * blockDim.x;
  auto group_sync = [] () {
    if (COOP) cg::this_grid().sync(); else cg::this_cluster().sync();
  };
  const int L = st->L, nl = 3 + 2 * L, epoch = st->epoch, pbase = st->pbase;
  int nm = b.pidx[line0];             /* matches of this scan so far: tracked identically by every thread */
  int ne = b.eidx[line0];
  /* exchanges done so far over the life of the filter: numbers the arrival epochs and alternates the two halves
   * of the exchange buffers (a per-scan count would let a fast rank overwrite a half a peer is still reading) */
  const int xseq0 = SHARD ? st->xseq : 0;
  int xdone = 0;
  double A[3][3], xp[3];              /* every thread's own copy of P[0:3,0:3] (mirrored) and x_pre */
  load_rr(g, b.top, A);
  xp[0] = st->x_pre[0]; xp[1] = st->x_pre[1]; xp[2] = st->x_pre[2];
  bool have_prev = false;             /* a matched line whose hot update has not been applied yet */
  int np_prev = 0;
  double pv0 = 0.0, pv1 = 0.0;        /* its innovation */
  double pS[4] = {0, 0, 0, 0};
  /* iteration `line1` only applies the last pending hot update */
  for (int line = line0; line <= line1; ++line) {
    const bool gating = line < line1;
    if (!gating && !have_prev) break;
    TS(0);
    /* ---- phase C of the previous match fused with phase A of this line ---- */
    double Rl[4] = {0, 0, 0, 0}, z0 = 0, z1 = 0;
    if (gating) {
      Rl[0] = R[4 * line]; Rl[1] = R[4 * line + 1]; Rl[2] = R[4 * line + 2]; Rl[3] = R[4 * line + 3];
      z0 = z[2 * line]; z1 = z[2 * line + 1];
    }
    const double2* Kv = b.Kp + (size_t)(own_slot0 + np_prev) * g.ld;
    const double2* KSv = b.KSp + (size_t)(own_slot0 + np_prev) * g.ld;
    double2 ks[3], kk[3];
    if (have_prev) {
      for (int r = 0; r < 3; ++r) { ks[r] = KSv[r]; kk[r] = Kv[r]; }
    }
    int cand = EKF_NO_MATCH;
    bool robot_done = !have_prev;
    for (int j = gtid; j < L; j += gstride) {
      const int a = 3 + 2 * j, bb = a + 1;
      double t0a = b.top[a], t0b = b.top[bb];
      double t1a = b.top[(size_t)g.ld + a], t1b = b.top[(size_t)g.ld + bb];
      double t2a = b.top[(size_t)2 * g.ld + a], t2b = b.top[(size_t)2 * g.ld + bb];
      double daa = b.diag[4 * j], dab = b.diag[4 * j + 1], dbb = b.diag[4 * j + 2];
      double ya = b.y[a], yb = b.y[bb];
      const int mt = b.matched[j];
      if (have_prev) {                                                /* Robot.cpp:564-589 on this landmark's hot elements */
        const double2 ka = Kv[a], kb = Kv[bb], ksa = KSv[a], ksb = KSv[bb];
        t0a = sub_rank2(t0a, ks[0], ka); t0b = sub_rank2(t0b, ks[0], kb);
        t1a = sub_rank2(t1a, ks[1], ka); t1b = sub_rank2(t1b, ks[1], kb);
        t2a = sub_rank2(t2a, ks[2], ka); t2b = sub_rank2(t2b, ks[2], kb);
        daa = sub_rank2(daa, ksa, ka); dab = sub_rank2(dab, ksa, kb); dbb = sub_rank2(dbb, ksb, kb);
        double ta = 0.0, tb = 0.0;
        axpy_skip(ta, ka.x, pv0); axpy_skip(ta, ka.y, pv1);
        axpy_skip(tb, kb.x, pv0); axpy_skip(tb, kb.y, pv1);
        ya = add_rn(ya, ta); yb = add_rn(yb, tb);
        b.top[a] = t0a; b.top[bb] = t0b;
        b.top[(size_t)g.ld + a] = t1a; b.top[(size_t)g.ld + bb] = t1b;
        b.top[(size_t)2 * g.ld + a] = t2a; b.top[(size_t)2 * g.ld + bb] = t2b;
        b.diag[4 * j] = daa; b.diag[4 * j + 1] = dab; b.diag[4 * j + 2] = dbb;
        b.y[a] = ya; b.y[bb] = yb;
      }
      if (!robot_done) { update_robot_block(kk, ks, pv0, pv1, A, xp); robot_done = true; }
      if (gating && cand == EKF_NO_MATCH && mt != epoch) {            /* Robot.cpp:313-501 */
        double Cm[5][5];
        for (int r = 0; r < 3; ++r) for (int q = 0; q < 3; ++q) Cm[r][q] = A[r][q];
        Cm[0][3] = Cm[3][0] = t0a; Cm[0][4] = Cm[4][0] = t0b;
        Cm[1][3] = Cm[3][1] = t1a; Cm[1][4] = Cm[4][1] = t1b;
        Cm[2][3] = Cm[3][2] = t2a; Cm[2][4] = Cm[4][2] = t2b;
        Cm[3][3] = daa; Cm[3][4] = Cm[4][3] = dab; Cm[4][4] = dbb;
        Gate G;
        gate_from_block(Cm, ya, yb, xp, z0, z1, Rl, G);
        if (G.singular) atomicMin(&b.jsing[line], j);                 /* reported by k_end_scan_a if below the winner */
        else if (!gate_rejects_d2(G.d2, g.gate_d2max)) { cand = j; gate_store(b.gates + (size_t)GATE_REC * j, G); }
      }
    }
    if (!robot_done) update_robot_block(kk, ks, pv0, pv1, A, xp);    /* threads without a landmark of their own */
    if (have_prev && gtid == 0) {     /* one writer publishes the robot block */
      for (int r = 0; r < 3; ++r) {
        for (int q = r; q < 3; ++q) b.top[(size_t)r * g.ld + q] = A[r][q];
        b.y[r] = xp[r]; st->pose[r] = xp[r]; st->x_pre[r] = xp[r];
      }
      st->v[0] = pv0; st->v[1] = pv1;
      for (int t = 0; t < 4; ++t) st->S[t] = pS[t];
    }
    if (!gating) break;
    TS(1);
    cand = __reduce_min_sync(0xffffffffu, cand);
    if ((threadIdx.x & 31) == 0) s_min[threadIdx.x >> 5] = cand;
    __syncthreads();
    if (threadIdx.x < 32) {
      int v = (threadIdx.x < FL_THREADS / 32) ? s_min[threadIdx.x] : EKF_NO_MATCH;
      v = __reduce_min_sync(0xffffffffu, v);
      if (threadIdx.x == 0 && v != EKF_NO_MATCH) atomicMin(&b.jbest[line], v);
    }
    TS(2);
    group_sync();                                                     /* hot state current, winner known */
    TS(3);
    const int j = b.jbest[line];
    const int np = nm - pbase;
    if (j == EKF_NO_MATCH) {                                          /* :309 / :325 / :493 */
      if (gtid == 0) { b.ext[ne] = line; b.eidx[line + 1] = ne + 1; b.pidx[line + 1] = nm; b.jout[line] = -1; }
      ne += 1;
      have_prev = false;
      continue;
    }
    /* ---- phase B: Robot.cpp:516-560 ---- */
    const int a = 3 + 2 * j, bb = a + 1;
    Gate G;
    gate_load(b.gates + (size_t)GATE_REC * j, G);
    /* the pending terms' entries at a and b are the same for every row: stage them once per CTA */
    const int npt = prev_cnt + np;
    PendingList pl;
    pl.prev_cnt = prev_cnt; pl.prev_slot0 = prev_slot0; pl.own_slot0 = own_slot0;
    for (int i = threadIdx.x; i < npt; i += blockDim.x) {
      const int slot = pl.slot(i);
      s_ka[i] = b.Kp[(size_t)slot * g.ld + a]; s_kb[i] = b.Kp[(size_t)slot * g.ld + bb];
      s_ksa[i] = b.KSp[(size_t)slot * g.ld + a]; s_ksb[i] = b.KSp[(size_t)slot * g.ld + bb];
    }
    GainRow d;
    int r = gtid;
    TS(4);
    if (!SHARD) {
      if (r < nl) gain_row_load(g, b, A, r, j, npt, pl, d);
      __syncthreads();
      TS(5);
      while (r < nl) {
        gain_row_correct(g, b, r, npt, d, pl, s_ka, s_kb, s_ksa, s_ksb);
        gain_row_emit(g, b, G, r, own_slot0 + np, d);
        r += gstride;
        if (r < nl) gain_row_load(g, b, A, r, j, npt, pl, d);
      }
    } else {
      /* part 1: every rank computes the current value of the cold slice entries it OWNS (row owner) and stores
       * them straight into every rank's exchange buffer over NVLink */
      const int xpar = (xseq0 + xdone) & 1;
      __syncthreads();
      for (; r < nl; r += gstride) {
        if (r <= 2 || r == a || r == bb) continue;                   /* hot entries are replicated */
        const int own_a = owner_of_row(g, min(r, a)), own_b = owner_of_row(g, min(r, bb));
        if (own_a != g.rank && own_b != g.rank) continue;
        double pa = 0.0, pb = 0.0;
        if (r < a) {                                                  /* P[r,a], P[r,b]: both in row r */
          const double* Pr = b.P + local_row(g, r) * g.ld;
          pa = Pr[a]; pb = Pr[bb];
          for (int i = 0; i < npt; ++i) {
            const double2 v = b.KSp[(size_t)pl.slot(i) * g.ld + r];
            pa = sub_rank2(pa, v, s_ka[i]); pb = sub_rank2(pb, v, s_kb[i]);
          }
        } else {                                                      /* P[a,r] (owner of row a), P[b,r] (owner of row b) */
          if (own_a == g.rank) pa = b.P[local_row(g, a) * g.ld + r];
          if (own_b == g.rank) pb = b.P[local_row(g, bb) * g.ld + r];
          for (int i = 0; i < npt; ++i) {
            const double2 v = b.Kp[(size_t)pl.slot(i) * g.ld + r];
            pa = sub_rank2(pa, s_ksa[i], v); pb = sub_rank2(pb, s_ksb[i], v);
          }
        }
        for (int p = 0; p < pe.world; ++p) {
          if (own_a == g.rank) xchg_col(pe, g, p, xpar, 0)[r] = pa;
          if (own_b == g.rank) xchg_col(pe, g, p, xpar, 1)[r] = pb;
        }
      }
      TS(8);
      __threadfence_system();
      group_sync();
      TS(9);
      if (gtid == 0) xgpu_exchange_barrier(pe, g, (unsigned long long)(xseq0 + xdone) + 1ull, &st->sticky);
      xdone += 1;
      TS(10);
      group_sync();
      TS(11);
      if (*(volatile int*)&st->sticky & EKF_STICKY_XCHG) {
        /* a peer never arrived: the gathered slices are stale.  No gain, no update: the remaining lines of the scan are
         * dropped (sane counters for the end-of-scan kernels) and the host marks the filter poisoned (EKF_ENCCL) */
        if (gtid == 0) for (int i = line; i < line1; ++i) { b.jout[i] = -1; b.pidx[i + 1] = nm; b.eidx[i + 1] = ne; }
        have_prev = false;
        break;
      }
      /* part 2: every rank forms the full K, K S (replicated) from the gathered slices */
      const double* cA = xchg_col(pe, g, g.rank, xpar, 0);
      const double* cB = xchg_col(pe, g, g.rank, xpar, 1);
      for (r = gtid; r < nl; r += gstride) {
        GainRow e;
        if (r <= 2) { e.p0 = A[r][0]; e.p1 = A[r][1]; e.p2 = A[r][2]; e.pa = b.top[(size_t)r * g.ld + a]; e.pb = b.top[(size_t)r * g.ld + bb]; }
        else {
          e.p0 = b.top[r]; e.p1 = b.top[(size_t)g.ld + r]; e.p2 = b.top[(size_t)2 * g.ld + r];
          if (r == a) { e.pa = b.diag[4 * j]; e.pb = b.diag[4 * j + 1]; }
          else if (r == bb) { e.pa = b.diag[4 * j + 1]; e.pb = b.diag[4 * j + 2]; }
          else { e.pa = __ldcg(cA + r); e.pb = __ldcg(cB + r); }
        }
        gain_row_emit(g, b, G, r, own_slot0 + np, e);
      }
    }
    if (gtid == 0) {                                                  /* :501-504 bookkeeping (read after the next barrier) */
      b.matched[j] = epoch;
      b.jout[line] = j;
      b.pidx[line + 1] = nm + 1; b.eidx[line + 1] = ne;
      st->np = np + 1;
    }
    TS(6);
    group_sync();                                                     /* K, K S complete */
    TS(7);
    have_prev = true;
    np_prev = np;
    nm += 1;
    pv0 = G.v[0]; pv1 = G.v[1];
    for (int t = 0; t < 4; ++t) pS[t] = G.S[t];
  }
  if (SHARD && gtid == 0) st->xseq = xseq0 + xdone;   /* every thread read xseq0 before the first barrier */
}

/* ------------------------------------------------------------------------------------------------ */
/* k_scan_lines2: the line loop with ONE barrier per line (single GPU; the row-sharded form stays on k_scan_lines).
 *
 * What made the first form need two barriers and several L2 round trips per line was the split of the work: landmarks
 * were gated by one thread, their gain rows formed by another, and the hot update of the next line waited for both.
 * Here a thread OWNS its landmarks (j = gtid, gtid + gstride, ...): their hot covariance entries (rows 0..2 of the two
 * columns, the 2x2 diagonal block), their state entries, AND their two gain rows.  The three robot rows of the gain are
 * formed redundantly by every thread from the 3x3 block it carries and the winner's six top entries, which travel with
 * the winner's gate record.  So after the one barrier that settles the first fit, a thread has everything it needs to
 * form its gain rows, apply the whole hot update to what it owns (Robot.cpp:564-602) and go straight to the next line's
 * gate: per line one barrier and one dependent round trip to L2 (the winner's record + the two column entries of the
 * owned rows) instead of two barriers and four.  While every thread owns at most one landmark (L <= threads: 8192 in
 * the cluster form, 10240 beside an overlapped sweep) the hot entries live in registers for the whole scan and memory
 * sees only write-through stores.  Same functions, same order of operations per element as k_scan_lines: identical bits
 * (test_all_launch_strategies_give_identical_bits). */
struct HotLm { double t0a, t0b, t1a, t1b, t2a, t2b, daa, dab, dbb, ya, yb; int mt; };
__device__ __forceinline__ void hot_load(const EkfGeom& g, const EkfBuffers& b, int j, HotLm& h) {
  const int a = 3 + 2 * j;
  h.t0a = b.top[a]; h.t0b = b.top[a + 1];
  h.t1a = b.top[(size_t)g.ld + a]; h.t1b = b.top[(size_t)g.ld + a + 1];
  h.t2a = b.top[(size_t)2 * g.ld + a]; h.t2b = b.top[(size_t)2 * g.ld + a + 1];
  h.daa = b.diag[4 * j]; h.dab = b.diag[4 * j + 1]; h.dbb = b.diag[4 * j + 2];
  h.ya = b.y[a]; h.yb = b.y[a + 1];
  h.mt = b.matched[j];
}
__device__ __forceinline__ void hot_store(const EkfGeom& g, const EkfBuffers& b, int j, const HotLm& h) {
  const int a = 3 + 2 * j;
  b.top[a] = h.t0a; b.top[a + 1] = h.t0b;
  b.top[(size_t)g.ld + a] = h.t1a; b.top[(size_t)g.ld + a + 1] = h.t1b;
  b.top[(size_t)2 * g.ld + a] = h.t2a; b.top[(size_t)2 * g.ld + a + 1] = h.t2b;
  b.diag[4 * j] = h.daa; b.diag[4 * j + 1] = h.dab; b.diag[4 * j + 2] = h.dbb;
  b.y[a] = h.ya; b.y[a + 1] = h.yb;
}

template <int FL_THREADS, bool COOP, bool CACHED>
__global__ void __launch_bounds__(FL_THREADS, 1) k_scan_lines2(EkfGeom g, EkfBuffers b, const double* __restrict__ z,
                                                               const double* __restrict__ R, int line0, int line1,
                                                               int own_slot0, int prev_slot0, const int* __restrict__ prev_cnt_ptr,
                                                               const double* __restrict__ pred_u, const double* __restrict__ pred_x, int pred_m,
                                                               const int* __restrict__ pred_carry) {
  __shared__ int s_min[FL_THREADS / 32];
  __shared__ double2 s_ka[FL_MAXP], s_kb[FL_MAXP], s_ksa[FL_MAXP], s_ksb[FL_MAXP];
  const int prev_cnt = prev_cnt_ptr ? *prev_cnt_ptr : 0;   /* previous scan's terms not yet folded into b.P */
  EkfDevState* st = b.st;
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x;
  const int gstride = gridDim.x * blockDim.x;
  const int scribe = gstride - 1;      /* the thread that writes the replicated results (last of the grid: on small maps it owns no landmark) */
  auto group_sync = [] () {
    if (COOP) cg::this_grid().sync(); else cg::this_cluster().sync();
  };
  if (pred_u) {                        /* the scan's prediction as the prologue of its (first) line-loop launch */
    predict_body(g, b, pred_u, pred_x, pred_m, gtid, gstride, pred_carry);
    __threadfence();
    group_sync();
  }
  const int L = st->L, epoch = st->epoch, pbase = st->pbase;
  int nm = b.pidx[line0];             /* matches of this scan so far: tracked identically by every thread */
  int ne = b.eidx[line0];
  double A[3][3], xp[3];              /* every thread's own copy of P[0:3,0:3] (mirrored) and x_pre */
  load_rr(g, b.top, A);
  xp[0] = st->x_pre[0]; xp[1] = st->x_pre[1]; xp[2] = st->x_pre[2];
  constexpr bool cached = CACHED;     /* host guarantee: at most one landmark per thread (L <= threads): its hot entries stay in registers */
  HotLm h;
  if (cached && gtid < L) hot_load(g, b, gtid, h);
  PendingList pl;
  pl.prev_cnt = prev_cnt; pl.prev_slot0 = prev_slot0; pl.own_slot0 = own_slot0;
  for (int line = line0; line < line1; ++line) {
    TS(0);
    /* ---- phase 1: gate of the owned landmarks (Robot.cpp:313-501) ---- */
    const double Rl[4] = {R[4 * line], R[4 * line + 1], R[4 * line + 2], R[4 * line + 3]};
    const double z0 = z[2 * line], z1 = z[2 * line + 1];
    int cand = EKF_NO_MATCH;
    for (int j = gtid; j < L; j += gstride) {
      if (!cached) hot_load(g, b, j, h);
      if (cand == EKF_NO_MATCH && h.mt != epoch) {
        double Cm[5][5];
        for (int r = 0; r < 3; ++r) for (int q = 0; q < 3; ++q) Cm[r][q] = A[r][q];
        Cm[0][3] = Cm[3][0] = h.t0a; Cm[0][4] = Cm[4][0] = h.t0b;
        Cm[1][3] = Cm[3][1] = h.t1a; Cm[1][4] = Cm[4][1] = h.t1b;
        Cm[2][3] = Cm[3][2] = h.t2a; Cm[2][4] = Cm[4][2] = h.t2b;
        Cm[3][3] = h.daa; Cm[3][4] = Cm[4][3] = h.dab; Cm[4][4] = h.dbb;
        Gate G;
        gate_from_block(Cm, h.ya, h.yb, xp, z0, z1, Rl, G);
        if (G.singular) atomicMin(&b.jsing[line], j);                 /* reported by k_end_scan_a if below the winner */
        else if (!gate_rejects_d2(G.d2, g.gate_d2max)) {
          cand = j;
          double* rec = b.gates + (size_t)GATE_REC * j;
          gate_store(rec, G);
          rec[14] = h.t0a; rec[15] = h.t0b; rec[16] = h.t1a; rec[17] = h.t1b; rec[18] = h.t2a; rec[19] = h.t2b;
        }
      }
    }
    TS(1);
    cand = __reduce_min_sync(0xffffffffu, cand);
    if ((threadIdx.x & 31) == 0) s_min[threadIdx.x >> 5] = cand;
    __syncthreads();
    if (threadIdx.x < 32) {
      int v = (threadIdx.x < FL_THREADS / 32) ? s_min[threadIdx.x] : EKF_NO_MATCH;
      v = __reduce_min_sync(0xffffffffu, v);
      if (threadIdx.x == 0 && v != EKF_NO_MATCH) atomicMin(&b.jbest[line], v);
    }
    TS(2);
    group_sync();                                                     /* the winner is known; last line's gains are visible */
    TS(3);
    const int jw = b.jbest[line];
    const int np = nm - pbase;
    if (jw != EKF_NO_MATCH) TS(8);
    if (jw == EKF_NO_MATCH) {                                         /* :309 / :325 / :493 */
      if (gtid == scribe) { b.ext[ne] = line; b.eidx[line + 1] = ne + 1; b.pidx[line + 1] = nm; b.jout[line] = -1; }
      ne += 1;
      continue;
    }
    /* ---- phase 2: gain rows (Robot.cpp:516-560) and the whole hot update (:564-602) of what this thread owns ---- */
    const int aw = 3 + 2 * jw, bw = aw + 1;
    const double* rec = b.gates + (size_t)GATE_REC * jw;
    Gate G;
    gate_load(rec, G);
    TS(9);
    const double wt[3][2] = {{rec[14], rec[15]}, {rec[16], rec[17]}, {rec[18], rec[19]}};   /* P[0..2, aw], P[0..2, bw] */
    const int npt = prev_cnt + np;
    for (int i = threadIdx.x; i < npt; i += blockDim.x) {            /* the pending terms' entries at aw, bw: once per CTA */
      const int slot = pl.slot(i);
      s_ka[i] = b.Kp[(size_t)slot * g.ld + aw]; s_kb[i] = b.Kp[(size_t)slot * g.ld + bw];
      s_ksa[i] = b.KSp[(size_t)slot * g.ld + aw]; s_ksb[i] = b.KSp[(size_t)slot * g.ld + bw];
    }
    const int out_slot = own_slot0 + np;
    double2 kk[3], ks[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) gain_row(G, A[r][0], A[r][1], A[r][2], wt[r][0], wt[r][1], kk[r], ks[r]);
    if (gtid == scribe) {
#pragma unroll
      for (int r = 0; r < 3; ++r) { b.Kp[(size_t)out_slot * g.ld + r] = kk[r]; b.KSp[(size_t)out_slot * g.ld + r] = ks[r]; }
    }
    TS(10);
    const double v0 = G.v[0], v1 = G.v[1];
    /* the two cold entries of each owned row (a, b) at the winner's columns, and the first pending terms' entries of
     * those rows: everything that has to come from L2 is issued here, in one round trip, before the staging barrier */
    constexpr int CH = 4;                                             /* pending terms fetched per row and round trip */
    const int jc = gtid;                                              /* cached form: the one owned landmark */
    const bool own1 = cached && jc < L;
    double cpa[2] = {0.0, 0.0}, cpb[2] = {0.0, 0.0};
    double2 cv[2][CH];
    int ckind = 0;
    if (own1 && jc != jw) {
      const int a = 3 + 2 * jc;
      ckind = jc < jw ? 1 : 2;
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        const int r = a + hf;
        if (ckind == 1) { cpa[hf] = b.P[(size_t)r * g.ld + aw]; cpb[hf] = b.P[(size_t)r * g.ld + bw]; }
        else { cpa[hf] = b.P[(size_t)aw * g.ld + r]; cpb[hf] = b.P[(size_t)bw * g.ld + r]; }
        const double2* src = ckind == 1 ? b.KSp : b.Kp;
#pragma unroll
        for (int t = 0; t < CH; ++t) if (t < npt) cv[hf][t] = src[(size_t)pl.slot(t) * g.ld + r];
      }
    }
    TS(11);
    __syncthreads();                                                  /* staging complete */
    TS(4);
    for (int j = gtid; j < L; j += gstride) {
      const int a = 3 + 2 * j, bb = a + 1;
      double2 Ka, KSa, Kb, KSb;
      if (cached) {
        /* rows a and b together: the pending terms in order, CH at a time (Robot.cpp:564-568 applied on the fly) */
        double pa0 = cpa[0], pb0 = cpb[0], pa1 = cpa[1], pb1 = cpb[1];
        if (j == jw) { pa0 = h.daa; pb0 = h.dab; pa1 = h.dab; pb1 = h.dbb; }
        else {
          const double2* src = ckind == 1 ? b.KSp : b.Kp;
          for (int i0 = 0; i0 < npt; i0 += CH) {
            if (i0 > 0) {
#pragma unroll
              for (int t = 0; t < CH; ++t) if (i0 + t < npt) {
                cv[0][t] = src[(size_t)pl.slot(i0 + t) * g.ld + a]; cv[1][t] = src[(size_t)pl.slot(i0 + t) * g.ld + bb];
              }
            }
#pragma unroll
            for (int t = 0; t < CH; ++t) if (i0 + t < npt) {
              if (ckind == 1) {
                pa0 = sub_rank2(pa0, cv[0][t], s_ka[i0 + t]); pb0 = sub_rank2(pb0, cv[0][t], s_kb[i0 + t]);
                pa1 = sub_rank2(pa1, cv[1][t], s_ka[i0 + t]); pb1 = sub_rank2(pb1, cv[1][t], s_kb[i0 + t]);
              } else {
                pa0 = sub_rank2(pa0, s_ksa[i0 + t], cv[0][t]); pb0 = sub_rank2(pb0, s_ksb[i0 + t], cv[0][t]);
                pa1 = sub_rank2(pa1, s_ksa[i0 + t], cv[1][t]); pb1 = sub_rank2(pb1, s_ksb[i0 + t], cv[1][t]);
              }
            }
          }
        }
        TS(12);
        gain_row(G, h.t0a, h.t1a, h.t2a, pa0, pb0, Ka, KSa);
        gain_row(G, h.t0b, h.t1b, h.t2b, pa1, pb1, Kb, KSb);
      } else {
        hot_load(g, b, j, h);
        /* several landmarks per thread: rows a and b one after the other through the chunked loader of the first form */
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int r = a + half;
          GainRow d;
          d.p0 = half ? h.t0b : h.t0a; d.p1 = half ? h.t1b : h.t1a; d.p2 = half ? h.t2b : h.t2a;
          d.kind = 0;
          if (j == jw) { d.pa = half ? h.dab : h.daa; d.pb = half ? h.dbb : h.dab; }
          else if (j < jw) {                                          /* column part: P[r, aw], P[r, bw] */
            const double* Pr = b.P + (size_t)r * g.ld;
            d.pa = Pr[aw]; d.pb = Pr[bw];
            d.kind = 1;
#pragma unroll
            for (int t = 0; t < 8; ++t) if (t < npt) d.v[t] = b.KSp[(size_t)pl.slot(t) * g.ld + r];
          } else {                                                    /* row part: P[aw, r], P[bw, r] */
            d.pa = b.P[(size_t)aw * g.ld + r]; d.pb = b.P[(size_t)bw * g.ld + r];
            d.kind = 2;
#pragma unroll
            for (int t = 0; t < 8; ++t) if (t < npt) d.v[t] = b.Kp[(size_t)pl.slot(t) * g.ld + r];
          }
          gain_row_correct(g, b, r, npt, d, pl, s_ka, s_kb, s_ksa, s_ksb);
          if (half) gain_row(G, d.p0, d.p1, d.p2, d.pa, d.pb, Kb, KSb);
          else gain_row(G, d.p0, d.p1, d.p2, d.pa, d.pb, Ka, KSa);
        }
      }
      TS(13);
      b.Kp[(size_t)out_slot * g.ld + a] = Ka; b.KSp[(size_t)out_slot * g.ld + a] = KSa;
      b.Kp[(size_t)out_slot * g.ld + bb] = Kb; b.KSp[(size_t)out_slot * g.ld + bb] = KSb;
      /* Robot.cpp:564-589 on this landmark's hot elements */
      h.t0a = sub_rank2(h.t0a, ks[0], Ka); h.t0b = sub_rank2(h.t0b, ks[0], Kb);
      h.t1a = sub_rank2(h.t1a, ks[1], Ka); h.t1b = sub_rank2(h.t1b, ks[1], Kb);
      h.t2a = sub_rank2(h.t2a, ks[2], Ka); h.t2b = sub_rank2(h.t2b, ks[2], Kb);
      h.daa = sub_rank2(h.daa, KSa, Ka); h.dab = sub_rank2(h.dab, KSa, Kb); h.dbb = sub_rank2(h.dbb, KSb, Kb);
      double ta = 0.0, tb = 0.0;
      axpy_skip(ta, Ka.x, v0); axpy_skip(ta, Ka.y, v1);
      axpy_skip(tb, Kb.x, v0); axpy_skip(tb, Kb.y, v1);
      h.ya = add_rn(h.ya, ta); h.yb = add_rn(h.yb, tb);
      if (j == jw) { h.mt = epoch; b.matched[j] = epoch; }            /* :501 */
      hot_store(g, b, j, h);                                          /* write-through: other kernels read the hot arrays */
    }
    TS(5);
    update_robot_block(kk, ks, v0, v1, A, xp);                        /* every thread's copy of the 3x3 block and the pose */
    if (gtid == scribe) {                                                  /* one writer publishes them; bookkeeping :501-504 */
      for (int r = 0; r < 3; ++r) {
        for (int q = r; q < 3; ++q) b.top[(size_t)r * g.ld + q] = A[r][q];
        b.y[r] = xp[r]; st->pose[r] = xp[r]; st->x_pre[r] = xp[r];
      }
      st->v[0] = v0; st->v[1] = v1;
      for (int t = 0; t < 4; ++t) st->S[t] = G.S[t];
      b.jout[line] = jw;
      b.pidx[line + 1] = nm + 1; b.eidx[line + 1] = ne;
      st->np = np + 1;
    }
    TS(6);
    nm += 1;
  }
}

/* after a sweep in the middle of a scan: the pending list restarts empty */
__global__ void k_flush_done(EkfBuffers b, int next_line) {
  if (blockIdx.x == 0 && threadIdx.x == 0) { b.st->pbase = b.pidx[next_line]; b.st->np = 0; }
}

/* between two chunks of an overlapped scan (lines [.., next_line) done): the snapshot the finished chunk's sweep will
 * need, then the pending list restarts empty for the next chunk */
__global__ void k_chunk_mark(EkfBuffers b, int next_line, EkfScanView* view) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    EkfDevState* st = b.st;
    view->cnt = b.pidx[next_line] - st->pbase; view->L = st->L;
    st->pbase = b.pidx[next_line]; st->np = 0;
  }
}

/* the map is empty (Robot.cpp:308-310): every line of the scan is queued */
__global__ void k_queue_all(EkfGeom g, EkfBuffers b, int m) {
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  for (int i = gid; i < m; i += gridDim.x * blockDim.x) {
    b.ext[i] = i; b.eidx[i + 1] = i + 1; b.pidx[i + 1] = 0; b.jout[i] = -1;
  }
}

/* ------------------------------------------------------------------------------------------------ */
/* THE roofline kernel.  Robot.cpp:564-568, P -= (K S) K', for the cold part of the upper triangle:
 * one pass that applies the scan's np pending rank-2 terms to every element in reference order.
 * 64x64 tiles; 8 warps x 8 rows; each lane owns two adjacent columns (one 16-byte load/store per row),
 * keeps its columns' K terms in registers (C terms at a time) and reads the rows' K S terms through
 * warp-uniform (broadcast) loads.  P is streamed with evict-first hints so K / KS stay in L2.
 * No masks: the stale copies of hot elements and the lower halves of diagonal tiles are swept too
 * (nothing reads them), so the kernel is a pure read-modify-write stream. */
struct TileId { int k, rb, cb; };

__device__ __forceinline__ long long tiles_before(int T, int rank, int world, long long k) {
  return k * (long long)(T - rank) - (long long)world * k * (k - 1) / 2;
}
__device__ __forceinline__ TileId decode_tile(int T, int rank, int world, long long idx) {
  const double A = (double)(T - rank) + 0.5 * world;
  double disc = A * A - 2.0 * world * (double)idx;
  if (disc < 0.0) disc = 0.0;
  long long k = (long long)((A - sqrt(disc)) / world);
  if (k < 0) k = 0;
  while (tiles_before(T, rank, world, k + 1) <= idx) ++k;
  while (k > 0 && tiles_before(T, rank, world, k) > idx) --k;
  TileId t;
  t.k = (int)k;
  t.rb = rank + world * (int)k;
  t.cb = t.rb + (int)(idx - tiles_before(T, rank, world, k));
  return t;
}

template <int C>
__global__ void __launch_bounds__(EKF_BLOCK, 2) k_sweep(EkfGeom g, EkfBuffers b, const int* __restrict__ np_ptr) {
  const int np = np_ptr ? *np_ptr : b.st->np;
  if (np <= 0) return;
  const int nl = 3 + 2 * b.st->L;
  const int T = (nl + EKF_TILE - 1) / EKF_TILE;
  if (g.rank >= T) return;
  const long long K_rows = (T - g.rank + g.world - 1) / g.world;
  const long long total = tiles_before(T, g.rank, g.world, K_rows);
  const long long idx = blockIdx.x;
  if (idx >= total) return;
  const TileId t = decode_tile(T, g.rank, g.world, idx);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r_base = t.rb * EKF_TILE + warp * 8;
  const int q = t.cb * EKF_TILE + 2 * lane;
  double* Pt = b.P + ((size_t)t.k * EKF_TILE + warp * 8) * g.ld + q;
  const int rows = min(8, nl - r_base);
  if (rows <= 0) return;
  double2 p[8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < rows) p[i] = __ldcs(reinterpret_cast<const double2*>(Pt + (size_t)i * g.ld));
  for (int c0 = 0; c0 < np; c0 += C) {
    double2 kq0[C], kq1[C];
#pragma unroll
    for (int c = 0; c < C; ++c)
      if (c0 + c < np) {
        const double2* Kc = b.Kp + (size_t)(c0 + c) * g.ld + q;
        kq0[c] = __ldg(Kc); kq1[c] = __ldg(Kc + 1);
      }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i < rows) {
#pragma unroll
        for (int c = 0; c < C; ++c)
          if (c0 + c < np) {
            const double2 ks = __ldg(b.KSp + (size_t)(c0 + c) * g.ld + r_base + i);
            p[i].x = sub_rank2(p[i].x, ks, kq0[c]);
            p[i].y = sub_rank2(p[i].y, ks, kq1[c]);
          }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < rows) __stcs(reinterpret_cast<double2*>(Pt + (size_t)i * g.ld), p[i]);
}

/* ------------------------------------------------------------------------------------------------ */
/* THE roofline kernel, pipelined form (the one the library launches).  Same arithmetic as k_sweep above,
 * organised for Blackwell: a persistent grid (one CTA per SM), one producer warp that streams 64x64 fp64
 * tiles of P (32 KB, TMA 2-D tensor copy) plus the matching 64-entry slices of the pending K and K S
 * terms (1 KB bulk copies) into a 4-deep shared-memory ring guarded by full/empty mbarriers, and eight
 * consumer warps that pull a tile into registers, apply the rank-2 terms in reference order and store
 * the result straight back to HBM with streaming stores.  The ring keeps ~190 KB per SM in flight, so
 * the fp64 work of a rank-2m update (m <= 8 per pass) hides under the HBM stream instead of serialising
 * with it.  No masks (see k_sweep). */
#define SW_C 8                        /* pending terms per pass */

template <int TR, int TC, int C>
struct __align__(128) SweepStage {
  double P[TR * TC];                  /* 32768 B, row-major TR x TC, written by TMA */
  double2 K[C][TC];                   /* K_c for the tile's columns */
  double2 KS[C][TR];                  /* (K S)_c for the tile's rows */
};
template <int TR, int TC, int STAGES, int C>
struct SweepShared {
  SweepStage<TR, TC, C> stage[STAGES];
  unsigned long long full[STAGES][2];  /* [stage][consumer group]: a group only ever waits on its own barrier (see k_sweep_quad) */
  unsigned long long empty[STAGES];
  unsigned long long emptyP[STAGES];   /* k_sweep_dmma: the stage's P tile alone is free again (its accumulators are in registers) */
  int meta[STAGES][4];                /* first local row, first global row, first column, - */
};

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_tile(void* dst, const CUtensorMap* map, int col, int row, unsigned long long* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(smem_u32(dst)), "l"((unsigned long long)map), "r"(smem_u32(bar)), "r"(col), "r"(row) : "memory");
}
/* same, with an L2 eviction-priority hint: the covariance is streamed once per sweep (evict first), so that
 * the small, constantly re-read hot state and pending lists are what stays in L2 */
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
  unsigned long long p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_load_tile_hint(void* dst, const CUtensorMap* map, int col, int row, unsigned long long* bar,
                                                   unsigned long long policy) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
               ::"r"(smem_u32(dst)), "l"((unsigned long long)map), "r"(smem_u32(bar)), "r"(col), "r"(row), "l"(policy) : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

/* The producer of both pipelined sweep kernels: ONE thread streams the CTA's tiles (and the matching slices of
 * the pending lists) into the shared-memory ring. */
template <int TR, int TC, int STAGES, int C, bool BOX8 = false>
__device__ __forceinline__ void sweep_producer(SweepShared<TR, TC, STAGES, C>& sh, const EkfGeom& g, const EkfBuffers& b,
                                               const CUtensorMap& tmapP, const CUtensorMap& tmapK, const CUtensorMap& tmapKS,
                                               int c0, int slot0, int np, int nl, unsigned long long* tile_counter, int sentinels) {
  const int T64 = (nl + EKF_TILE - 1) / EKF_TILE;      /* 64-row ownership blocks in the live part */
  const int Tc = (nl + TC - 1) / TC;                   /* tile columns */
  constexpr int SUB = EKF_TILE / TR;                   /* sub-row blocks per ownership block */
  /* more than 4 pending terms: ONE 2-D TMA copy fetches the 8-slot band of K (resp. K S) for the tile's
   * columns (rows) -- 3 TMA operations per tile instead of 17 */
  const bool band = np > 4;
  const int nbands = (np + 7) / 8;
  const unsigned long long pol = l2_policy_evict_first();
  const unsigned bytes = TR * TC * sizeof(double) + (unsigned)(band ? 8 * nbands : np) * (TC + TR) * sizeof(double2);
  int k = 0;                                        /* local ownership block */
  int gb = g.rank;                                  /* its global index */
  long long base = 0;                               /* index of the block's first tile */
  int cb0 = (EKF_TILE * gb) / TC;
  long long cnt = (gb < T64) ? (long long)SUB * (Tc - cb0) : 0;
  int it = 0;
  /* tiles are handed out by a global counter (zeroed before the launch): CTAs that share their SM with
   * another kernel simply take fewer tiles.  The indices a CTA draws are increasing, which is all the
   * incremental decode needs.  tile_counter == NULL: static round robin. */
  for (long long idx = tile_counter ? (long long)atomicAdd(tile_counter, 1ull) : (long long)blockIdx.x; gb < T64;
       idx = tile_counter ? (long long)atomicAdd(tile_counter, 1ull) : idx + gridDim.x, ++it) {
    while (gb < T64 && idx >= base + cnt) {
      base += cnt; ++k; gb += g.world;
      cb0 = (EKF_TILE * gb) / TC;
      cnt = (gb < T64) ? (long long)SUB * (Tc - cb0) : 0;
    }
    if (gb >= T64) break;
    const int rem = (int)(idx - base);
    const int sub = rem / (Tc - cb0), cb = cb0 + rem % (Tc - cb0);
    const int lrow0 = k * EKF_TILE + sub * TR, grow0 = gb * EKF_TILE + sub * TR, col0 = cb * TC;
    const int s = it % STAGES;
    const unsigned ph = (it / STAGES) & 1;
    mbar_wait(&sh.empty[s], ph ^ 1);
    sh.meta[s][0] = lrow0; sh.meta[s][1] = grow0; sh.meta[s][2] = col0; sh.meta[s][3] = 1;
    unsigned long long* fullb = &sh.full[s][sentinels > 1 ? (it & 1) : 0];     /* the barrier of the group that consumes tile `it` */
    mbar_expect_tx(fullb, bytes);
    if (BOX8) {
      /* the tile as eight 64-row x 8-column boxes, each dense in shared memory (row pitch 64 B): the layout the
       * tensor-core consumers read their 8x8 accumulator fragments from without bank conflicts (k_sweep_dmma) */
#pragma unroll
      for (int bx = 0; bx < TC / 8; ++bx) tma_load_tile_hint(sh.stage[s].P + bx * TR * 8, &tmapP, col0 + 8 * bx, lrow0, fullb, pol);
    } else {
      tma_load_tile_hint(sh.stage[s].P, &tmapP, col0, lrow0, fullb, pol);
    }
    if (band) {
      for (int bi = 0; bi < nbands; ++bi) {
        tma_load_tile(sh.stage[s].K[8 * bi], &tmapK, 2 * col0, slot0 + c0 + 8 * bi, fullb);
        tma_load_tile(sh.stage[s].KS[8 * bi], &tmapKS, 2 * grow0, slot0 + c0 + 8 * bi, fullb);
      }
    } else {
      for (int c = 0; c < np; ++c) {
        bulk_load(sh.stage[s].K[c], b.Kp + (size_t)(slot0 + c0 + c) * g.ld + col0, TC * sizeof(double2), fullb);
        bulk_load(sh.stage[s].KS[c], b.KSp + (size_t)(slot0 + c0 + c) * g.ld + grow0, TR * sizeof(double2), fullb);
      }
    }
  }
  /* tell the consumers there is nothing more: `sentinels` stages with valid = 0 (one per consumer group) */
  for (int e = 0; e < sentinels; ++e, ++it) {
    const int s = it % STAGES;
    const unsigned ph = (it / STAGES) & 1;
    mbar_wait(&sh.empty[s], ph ^ 1);
    sh.meta[s][3] = 0;
    mbar_arrive(&sh.full[s][sentinels > 1 ? (it & 1) : 0]);
  }
}

/* The producer of the tensor-core sweep.  Same tile order and ring as sweep_producer, but a stage is refilled in TWO steps:
 * its P tile as soon as the consuming group has the accumulators in registers (barrier emptyP: right at the start of the
 * group's work on the previous occupant), its K / K S bands when that group is done with them (barrier empty).  The P tile
 * is the part that comes from HBM; with the two-stage ring of the 32-term pass a stage used to be refilled only after its
 * group had finished, so every tile's HBM round trip was exposed (tensor pipe 70 % active).  The producer runs one tile
 * ahead: P of tile it + 1 is requested before the bands of tile it. */
template <int STAGES, int C>
__device__ __forceinline__ void sweep_producer_split(SweepShared<64, 64, STAGES, C>& sh, const EkfGeom& g,
                                                     const CUtensorMap& tmapP, const CUtensorMap& tmapK, const CUtensorMap& tmapKS,
                                                     int c0, int slot0, int np, int nl, unsigned long long* tile_counter) {
  constexpr int TR = 64, TC = 64;
  const int T64 = (nl + EKF_TILE - 1) / EKF_TILE;
  const int Tc = (nl + TC - 1) / TC;
  const int nbands = (np + 7) / 8;
  const unsigned long long pol = l2_policy_evict_first();
  const unsigned bytes = TR * TC * sizeof(double) + (unsigned)(8 * nbands) * (TC + TR) * sizeof(double2);
  int k = 0, gb = g.rank;
  long long base = 0;
  int cb0 = (EKF_TILE * gb) / TC;
  long long cnt = (gb < T64) ? (long long)(Tc - cb0) : 0;
  long long idx = tile_counter ? (long long)atomicAdd(tile_counter, 1ull) : (long long)blockIdx.x;
  /* decode of the next tile this CTA draws (indices increase: incremental) */
  auto next_tile = [&](int& lrow0, int& grow0, int& col0) -> bool {
    while (gb < T64 && idx >= base + cnt) {
      base += cnt; ++k; gb += g.world;
      cb0 = (EKF_TILE * gb) / TC;
      cnt = (gb < T64) ? (long long)(Tc - cb0) : 0;
    }
    if (gb >= T64) return false;
    const int rem = (int)(idx - base);
    lrow0 = k * EKF_TILE; grow0 = gb * EKF_TILE; col0 = (cb0 + rem) * TC;
    idx = tile_counter ? (long long)atomicAdd(tile_counter, 1ull) : idx + gridDim.x;
    return true;
  };
  auto issue_p = [&](int it, int lrow0, int grow0, int col0) {
    const int s = it % STAGES;
    const unsigned ph = (it / STAGES) & 1;
    mbar_wait(&sh.emptyP[s], ph ^ 1);
    sh.meta[s][0] = lrow0; sh.meta[s][1] = grow0; sh.meta[s][2] = col0; sh.meta[s][3] = 1;
    unsigned long long* fullb = &sh.full[s][it & 1];
    mbar_expect_tx(fullb, bytes);                      /* the whole stage: the phase completes only once the bands have landed too */
#pragma unroll
    for (int bx = 0; bx < TC / 8; ++bx) tma_load_tile_hint(sh.stage[s].P + bx * TR * 8, &tmapP, col0 + 8 * bx, lrow0, fullb, pol);
  };
  auto issue_bands = [&](int it, int grow0, int col0) {
    const int s = it % STAGES;
    const unsigned ph = (it / STAGES) & 1;
    mbar_wait(&sh.empty[s], ph ^ 1);
    unsigned long long* fullb = &sh.full[s][it & 1];
    for (int bi = 0; bi < nbands; ++bi) {
      tma_load_tile(sh.stage[s].K[8 * bi], &tmapK, 2 * col0, slot0 + c0 + 8 * bi, fullb);
      tma_load_tile(sh.stage[s].KS[8 * bi], &tmapKS, 2 * grow0, slot0 + c0 + 8 * bi, fullb);
    }
  };
  int lr = 0, gr = 0, cc = 0, it = 0;
  bool have = next_tile(lr, gr, cc);
  if (have) issue_p(0, lr, gr, cc);
  while (have) {
    int lr2 = 0, gr2 = 0, cc2 = 0;
    const bool have2 = next_tile(lr2, gr2, cc2);
    if (have2) issue_p(it + 1, lr2, gr2, cc2);
    issue_bands(it, gr, cc);
    lr = lr2; gr = gr2; cc = cc2; have = have2; ++it;
  }
  for (int e = 0; e < 2; ++e, ++it) {                   /* one sentinel per consumer group */
    const int s = it % STAGES;
    const unsigned ph = (it / STAGES) & 1;
    mbar_wait(&sh.emptyP[s], ph ^ 1);
    mbar_wait(&sh.empty[s], ph ^ 1);
    sh.meta[s][3] = 0;
    mbar_arrive(&sh.full[s][it & 1]);
  }
}

/* Tiles are TR rows x TC columns (TR*TC = 4096 doubles = 32 KB; TR <= 64 <= TC).  The upper triangle is
 * covered by, for each 64-row ownership block gb (this rank's: gb = rank + world*k), the 64/TR sub-row
 * blocks times the tile columns cb >= floor(64*gb / TC).  Tiles are numbered in that order; the
 * producer walks its tiles in increasing order, so it decodes incrementally (no division, no sqrt). */
/* C = pending terms applied per pass (8, 16 or 32).  Up to ~16 terms the pass stays HBM-bound (8 terms keep the
 * fp64 pipe 34 % busy); 32 terms are fp64-issue-bound (~1.35x the HBM time) -- still far cheaper than four
 * HBM-bound passes of 8.  The ring shrinks with C (4 / 3 / 2 stages) to stay inside 227 KB. */
template <int TR, int TC, int STAGES, int CW, int C>
__global__ void __launch_bounds__((CW + 1) * 32, 1)
k_sweep_pipe(EkfGeom g, EkfBuffers b, const __grid_constant__ CUtensorMap tmapP, const __grid_constant__ CUtensorMap tmapK,
             const __grid_constant__ CUtensorMap tmapKS, double* __restrict__ dst, int c0,
             int slot0, const EkfScanView* __restrict__ view, unsigned long long* __restrict__ tile_counter) {
  typedef SweepShared<TR, TC, STAGES, C> Shared;
  extern __shared__ unsigned char sw_raw[];
  /* TMA destinations want 128-byte alignment; the launcher over-allocates by 1 KB for this round-up */
  Shared& sh = *reinterpret_cast<Shared*>(sw_raw + ((1024u - (smem_u32(sw_raw) & 1023u)) & 1023u));
  /* view != NULL: the scan's own snapshot (its sweep may run while the next scan already changes st);
   * the out-of-place form (dst != source) must run even with no pending term: it is then a copy */
  const int np_all = view ? view->cnt : b.st->np;
  const int np = max(0, min(C, np_all - c0));
  if (np <= 0 && (dst == b.P || c0 > 0)) return;
  const int nl = 3 + 2 * (view ? view->L : b.st->L);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&sh.full[s][0], 1); mbar_init(&sh.empty[s], CW); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (warp == CW) {
    if (lane == 0) sweep_producer<TR, TC, STAGES, C>(sh, g, b, tmapP, tmapK, tmapKS, c0, slot0, np, nl, tile_counter, 1);
    return;
  }
  /* ---------------- consumers ---------------- */
  constexpr int WPR = TC / 64;                          /* warps across one tile row */
  constexpr int RPP = CW / WPR;                         /* rows per pass */
  constexpr int PT = TR / RPP;                          /* rows per thread */
  const int ccol = ((warp % WPR) * 32 + lane) * 2;      /* this lane's two columns inside the tile */
  const int crow = warp / WPR;
  for (int it = 0;; ++it) {
    const int s = it % STAGES;
    const unsigned ph = (it / STAGES) & 1;
    mbar_wait(&sh.full[s][0], ph);
    if (!sh.meta[s][3]) break;
    const SweepStage<TR, TC, C>& st = sh.stage[s];
    const int lrow0 = sh.meta[s][0], grow0 = sh.meta[s][1], col0 = sh.meta[s][2];
    double2 p[PT];
#pragma unroll
    for (int i = 0; i < PT; ++i) p[i] = *reinterpret_cast<const double2*>(&st.P[(crow + i * RPP) * TC + ccol]);
    for (int c = 0; c < np; ++c) {
      const double2 kq0 = st.K[c][ccol], kq1 = st.K[c][ccol + 1];
#pragma unroll
      for (int i = 0; i < PT; ++i) {
        const double2 ks = st.KS[c][crow + i * RPP];
        p[i].x = sub_rank2(p[i].x, ks, kq0);
        p[i].y = sub_rank2(p[i].y, ks, kq1);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&sh.empty[s]);
    double* Pt = dst + ((size_t)lrow0 + crow) * g.ld + (size_t)col0 + ccol;
    if (grow0 + TR <= nl && col0 + TC <= nl) {
#pragma unroll
      for (int i = 0; i < PT; ++i) __stcs(reinterpret_cast<double2*>(Pt + (size_t)(i * RPP) * g.ld), p[i]);
    } else {
      /* edge tile: dead rows / columns are left alone -- the line stream may be appending landmarks there
       * (augmentation) while this sweep is still in flight */
      const int q = col0 + ccol;
#pragma unroll
      for (int i = 0; i < PT; ++i) {
        if (grow0 + crow + i * RPP < nl) {
          if (q + 1 < nl) __stcs(reinterpret_cast<double2*>(Pt + (size_t)(i * RPP) * g.ld), p[i]);
          else if (q < nl) Pt[(size_t)(i * RPP) * g.ld] = p[i].x;
        }
      }
    }
  }
}

/* ------------------------------------------------------------------------------------------------ */
/* k_sweep_quad: the form of the pipelined sweep the library launches by default.  Same ring, same producer, same
 * per-element arithmetic and order as k_sweep_pipe<64,64,...>; what changes is how the consumers hold a tile.
 *
 * ncu on k_sweep_pipe at 8 pending terms (profiles/r1_ncu_sweep_pipe.csv): the LSU data pipe is 92 % busy and
 * shared-memory wavefronts are at 82 % of peak while DRAM sits at 74 % -- the kernel is bound by shared-memory
 * operand delivery, not by HBM: each lane owns 8 rows x 2 columns, so every term costs 8 warp-uniform LDS.128
 * (K S of a row: 2 wavefronts each) plus 2 LDS.128 of its columns' K that hit a 2-way bank conflict (stride
 * 32 B), i.e. 34 wavefronts per 32 DFMA instructions.
 *
 * Here a lane owns 8 rows x 4 columns (two 16-byte column pairs 32 columns apart): a HALF-warp spans the 64
 * columns of a tile row, the two halves of a warp take different rows, a warp covers 16 rows and FOUR warps
 * cover the tile; the eight consumer warps form two groups that take alternate ring stages.  Per term and
 * warp: 8 LDS.128 of K S (uniform per half-warp, each now feeding 8 DFMAs instead of 4) + 4 LDS.128 of K made
 * conflict-free by letting lanes 4..7 of every 8 fetch their pair in the opposite order (then swapped back in
 * registers): 24 wavefronts per 64 DFMA instructions -- 2.8x less shared-memory traffic per flop. */
template <int STAGES, int C>
__global__ void __launch_bounds__(9 * 32, 1)
k_sweep_quad(EkfGeom g, EkfBuffers b, const __grid_constant__ CUtensorMap tmapP, const __grid_constant__ CUtensorMap tmapK,
             const __grid_constant__ CUtensorMap tmapKS, double* __restrict__ dst, int c0,
             int slot0, const EkfScanView* __restrict__ view, unsigned long long* __restrict__ tile_counter) {
  constexpr int TR = 64, TC = 64, CW = 8;
  typedef SweepShared<TR, TC, STAGES, C> Shared;
  extern __shared__ unsigned char sw_raw[];
  Shared& sh = *reinterpret_cast<Shared*>(sw_raw + ((1024u - (smem_u32(sw_raw) & 1023u)) & 1023u));
  const int np_all = view ? view->cnt : b.st->np;
  const int np = max(0, min(C, np_all - c0));
  if (np <= 0 && (dst == b.P || c0 > 0)) return;
  const int nl = 3 + 2 * (view ? view->L : b.st->L);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&sh.full[s][0], 1); mbar_init(&sh.full[s][1], 1); mbar_init(&sh.empty[s], CW / 2); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (warp == CW) {
    if (lane == 0) sweep_producer<TR, TC, STAGES, C>(sh, g, b, tmapP, tmapK, tmapKS, c0, slot0, np, nl, tile_counter, 2);
    return;
  }
  /* ---------------- consumers: 2 groups x 4 warps ---------------- */
  const int grp = warp >> 2;
  const int l16 = lane & 15;
  const int row0 = 16 * (warp & 3) + 8 * (lane >> 4);        /* this lane's 8 rows inside the tile */
  const int cA = 2 * l16, cB = 32 + 2 * l16;                 /* its two column pairs */
  const bool sw = (l16 & 4) != 0;                            /* fetch the pair's halves in the opposite order */
  const int o0 = sw ? 1 : 0, o1 = sw ? 0 : 1;
  /* Each (stage, group) pair has its OWN full barrier.  mbarrier waits see only a phase PARITY; with an odd ring a
   * stage alternates between the groups, and a group that ran ahead could mistake the other group's not-yet-landed
   * tile for its own (same parity) if they shared the barrier.  With its own barrier a group observes every phase
   * of it in order: the k-th use of (stage, group) is tile k * PERIOD + ... , PERIOD = lcm(STAGES, 2). */
  constexpr int PERIOD = (STAGES % 2) ? 2 * STAGES : STAGES;
  for (int it = grp;; it += 2) {
    const int s = it % STAGES;
    const unsigned ph = (it / PERIOD) & 1;
    mbar_wait(&sh.full[s][grp], ph);
    if (!sh.meta[s][3]) break;
    const SweepStage<TR, TC, C>& st = sh.stage[s];
    const int lrow0 = sh.meta[s][0], grow0 = sh.meta[s][1], col0 = sh.meta[s][2];
    double2 pa[8], pb[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      pa[i] = *reinterpret_cast<const double2*>(&st.P[(row0 + i) * TC + cA]);
      pb[i] = *reinterpret_cast<const double2*>(&st.P[(row0 + i) * TC + cB]);
    }
#pragma unroll (C > 8 ? 4 : 2)
    for (int c = 0; c < np; ++c) {
      const double2 a0 = st.K[c][cA + o0], a1 = st.K[c][cA + o1];
      const double2 b0 = st.K[c][cB + o0], b1 = st.K[c][cB + o1];
      const double2 ka0 = sw ? a1 : a0, ka1 = sw ? a0 : a1;
      const double2 kb0 = sw ? b1 : b0, kb1 = sw ? b0 : b1;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const double2 ks = st.KS[c][row0 + i];
        pa[i].x = sub_rank2(pa[i].x, ks, ka0);
        pa[i].y = sub_rank2(pa[i].y, ks, ka1);
        pb[i].x = sub_rank2(pb[i].x, ks, kb0);
        pb[i].y = sub_rank2(pb[i].y, ks, kb1);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&sh.empty[s]);
    double* Pt = dst + ((size_t)lrow0 + row0) * g.ld + (size_t)col0;
    if (grow0 + TR <= nl && col0 + TC <= nl) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        __stcs(reinterpret_cast<double2*>(Pt + (size_t)i * g.ld + cA), pa[i]);
        __stcs(reinterpret_cast<double2*>(Pt + (size_t)i * g.ld + cB), pb[i]);
      }
    } else {
      /* edge tile: dead rows / columns are left alone (see k_sweep_pipe) */
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (grow0 + row0 + i < nl) {
          double* Pr = Pt + (size_t)i * g.ld;
          const int qa = col0 + cA, qb = col0 + cB;
          if (qa + 1 < nl) __stcs(reinterpret_cast<double2*>(Pr + cA), pa[i]); else if (qa < nl) Pr[cA] = pa[i].x;
          if (qb + 1 < nl) __stcs(reinterpret_cast<double2*>(Pr + cB), pb[i]); else if (qb < nl) Pr[cB] = pb[i].x;
        }
      }
    }
  }
}

/* ------------------------------------------------------------------------------------------------ */
/* k_sweep_dmma: the same pass on the fp64 tensor cores (north_star: "DMMA only if batched observations make the update a
 * genuine dense contraction" -- from ~12 pending terms on the DFMA form above is bound by fp64 issue and shared-memory
 * operand delivery, not by HBM).  P_tile(64x64) -= KS_tile(64 x 2m) * K_tile'(2m x 64) as mma.sync.m8n8k4.f64:
 *   A[row][k]  = -(K S)_{c + k/2}[row].{x, y}      B[k][col] = K_{c + k/2}[col].{x, y}      k = 0..3: two pending terms
 * Measured on B200 (scripts/dmma_probe.cu, profiles/r2_dmma_probe.log): the instruction accumulates as the chain
 * d = fma(a_k, b_k, d), k = 0..3 in order, one rounding per step -- bit for bit sub_rank2() applied term after term -- at
 * 37 TFLOP/s against 34 for DFMA, with 8x fewer issue slots per flop and operands that stay in registers across 16 MMAs.
 * Same ring and producer as k_sweep_quad; the producer lands the P tile as eight 64 x 8 boxes (row pitch 64 B) so that
 * a warp's accumulator-fragment load -- lane (g, t) takes row g, columns 2t, 2t+1 of an 8x8 block -- is one conflict-free
 * LDS.128.  A warp owns 16 rows x 64 columns: 2 x 8 blocks, 32 doubles per lane; per two terms it loads 2 + 8 operand
 * words and issues 16 MMAs. */
__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}
template <int STAGES, int C, bool SPLIT>
__global__ void __launch_bounds__(9 * 32, 1)
k_sweep_dmma(EkfGeom g, EkfBuffers b, const __grid_constant__ CUtensorMap tmapP, const __grid_constant__ CUtensorMap tmapK,
             const __grid_constant__ CUtensorMap tmapKS, double* __restrict__ dst, int c0,
             int slot0, const EkfScanView* __restrict__ view, unsigned long long* __restrict__ tile_counter) {
  constexpr int TR = 64, TC = 64, CW = 8;
  typedef SweepShared<TR, TC, STAGES, C> Shared;
  extern __shared__ unsigned char sw_raw[];
  Shared& sh = *reinterpret_cast<Shared*>(sw_raw + ((1024u - (smem_u32(sw_raw) & 1023u)) & 1023u));
  const int np_all = view ? view->cnt : b.st->np;
  const int np = max(0, min(C, np_all - c0));
  if (np <= 0 && (dst == b.P || c0 > 0)) return;
  const int nl = 3 + 2 * (view ? view->L : b.st->L);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&sh.full[s][0], 1); mbar_init(&sh.full[s][1], 1); mbar_init(&sh.empty[s], CW / 2); mbar_init(&sh.emptyP[s], CW / 2);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (warp == CW) {
    if (lane == 0) {
      /* the split refill needs the band copies (more than 4 terms: always the case where this kernel is selected) */
      if (SPLIT && np > 4) sweep_producer_split<STAGES, C>(sh, g, tmapP, tmapK, tmapKS, c0, slot0, np, nl, tile_counter);
      else sweep_producer<TR, TC, STAGES, C, true>(sh, g, b, tmapP, tmapK, tmapKS, c0, slot0, np, nl, tile_counter, 2);
    }
    return;
  }
  const bool split = SPLIT && np > 4;
  /* ---------------- consumers: 2 groups x 4 warps, a warp = rows 16 (warp & 3) .. + 15 of the tile ---------------- */
  const int grp = warp >> 2;
  const int gq = lane >> 2, tq = lane & 3;                   /* fragment coordinates of this lane */
  const int row0 = 16 * (warp & 3) + gq;                     /* its rows: row0, row0 + 8 */
  const int comp = tq & 1, tsel = tq >> 1;                   /* operand word: component x / y of term (k0 + tsel) */
  constexpr int PERIOD = (STAGES % 2) ? 2 * STAGES : STAGES;
  for (int it = grp;; it += 2) {
    const int s = it % STAGES;
    const unsigned ph = (it / PERIOD) & 1;
    mbar_wait(&sh.full[s][grp], ph);
    if (!sh.meta[s][3]) break;
    const SweepStage<TR, TC, C>& st = sh.stage[s];
    const int lrow0 = sh.meta[s][0], grow0 = sh.meta[s][1], col0 = sh.meta[s][2];
    double2 acc[2][8];
#pragma unroll
    for (int mb = 0; mb < 2; ++mb)
#pragma unroll
      for (int nb = 0; nb < 8; ++nb)
        acc[mb][nb] = *reinterpret_cast<const double2*>(&st.P[(nb * TR + row0 + 8 * mb) * 8 + 2 * tq]);
    if (split) {                                               /* the P tile may be refilled: its HBM round trip runs under the MMAs */
      __syncwarp();
      if (lane == 0) mbar_arrive(&sh.emptyP[s]);
    }
    const double* KSw = reinterpret_cast<const double*>(&st.KS[0][0]);
    const double* Kw = reinterpret_cast<const double*>(&st.K[0][0]);
#pragma unroll 2
    for (int k0 = 0; k0 < np; k0 += 2) {
      const int term = k0 + tsel;
      const bool valid = term < np;                          /* odd count: the last step's second term is zero */
      double a[2], bq[8];
#pragma unroll
      for (int mb = 0; mb < 2; ++mb) a[mb] = valid ? -KSw[(term * TR + row0 + 8 * mb) * 2 + comp] : 0.0;
#pragma unroll
      for (int nb = 0; nb < 8; ++nb) bq[nb] = valid ? Kw[(term * TC + 8 * nb + gq) * 2 + comp] : 0.0;
#pragma unroll
      for (int mb = 0; mb < 2; ++mb)
#pragma unroll
        for (int nb = 0; nb < 8; ++nb) dmma884(acc[mb][nb].x, acc[mb][nb].y, a[mb], bq[nb]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&sh.empty[s]);
    double* Pt = dst + ((size_t)lrow0 + row0) * g.ld + (size_t)col0 + 2 * tq;
    if (grow0 + TR <= nl && col0 + TC <= nl) {
#pragma unroll
      for (int mb = 0; mb < 2; ++mb)
#pragma unroll
        for (int nb = 0; nb < 8; ++nb) __stcs(reinterpret_cast<double2*>(Pt + (size_t)(8 * mb) * g.ld + 8 * nb), acc[mb][nb]);
    } else {
      /* edge tile: dead rows / columns are left alone (see k_sweep_pipe) */
#pragma unroll
      for (int mb = 0; mb < 2; ++mb) {
        if (grow0 + row0 + 8 * mb < nl) {
          double* Pr = Pt + (size_t)(8 * mb) * g.ld;
#pragma unroll
          for (int nb = 0; nb < 8; ++nb) {
            const int q = col0 + 8 * nb + 2 * tq;
            if (q + 1 < nl) __stcs(reinterpret_cast<double2*>(Pr + 8 * nb), acc[mb][nb]); else if (q < nl) Pr[8 * nb] = acc[mb][nb].x;
          }
        }
      }
    }
  }
}

/* ------------------------------------------------------------------------------------------------ */
/* Robot.cpp:702-716 then :776-866 phase A (per unmatched line: world-frame parameters, P_ll, and the
 * rows 0..2 of its new columns -- all functions of the 3x3 robot block only). */
__global__ void __launch_bounds__(512) k_end_scan_a(EkfGeom g, EkfBuffers b, const double* __restrict__ z, const double* __restrict__ R, int m,
                                                    int slot0, EkfScanView* view, int prev_slot0, const int* __restrict__ prev_cnt_ptr) {
  EkfDevState* st = b.st;
  __shared__ double s_pose[3];
  __shared__ double s_y01[2];
  if (threadIdx.x == 0) {
    if (m == 0 || b.pidx[m] == 0) {                                   /* :702-716 */
      b.y[0] = st->x_pre[0]; b.y[1] = st->x_pre[1]; b.y[2] = st->x_pre[2];
      double th = st->x_pre[2];
      normalize_radian(th);
      st->pose[0] = st->x_pre[0]; st->pose[1] = st->x_pre[1]; st->pose[2] = th;
    }
    s_pose[0] = st->pose[0]; s_pose[1] = st->pose[1]; s_pose[2] = st->pose[2];
    s_y01[0] = b.y[0]; s_y01[1] = b.y[1];
  }
  __syncthreads();
  const int ne = b.eidx[m];
  const int L = st->L;
  const int n_add = min(ne, g.cap - L);
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    st->n_added = n_add;
    if (n_add < ne) atomicOr(&st->sticky, EKF_STICKY_CAPACITY);       /* the reference overruns y[] here (Q4) */
  }
  {     /* EKF_ESINGULAR: some line's first fit skipped a singular pair before its winner (any, when it matched nothing) */
    int skipped = 0;
    for (int i = threadIdx.x; i < m; i += blockDim.x) skipped |= b.jsing[i] < b.jbest[i];
    if (__syncthreads_or(skipped) && threadIdx.x == 0) atomicOr(&st->sticky, EKF_STICKY_SINGULAR);
  }
  /* this scan's pending terms have no entry for the rows being appended: zero them, so that the (possibly
   * later) sweep and the next scan's on-the-fly corrections see K = 0 there */
  /* prev_cnt_ptr != NULL (a sweep group stays open): the same for the terms of the previous group, which the group's next
   * scan still corrects against -- a term contributes exactly zero at every row appended after it was formed */
  {
    const int cnt = b.pidx[m] - st->pbase, r0 = 3 + 2 * L, r1 = 3 + 2 * (L + n_add);
    const int pcnt = prev_cnt_ptr ? *prev_cnt_ptr : 0;
    for (int i = 0; i < cnt + pcnt; ++i) {
      const size_t slot = i < cnt ? slot0 + i : prev_slot0 + (i - cnt);
      for (int r = r0 + threadIdx.x; r < r1; r += blockDim.x) {
        b.Kp[slot * g.ld + r] = make_double2(0.0, 0.0);
        b.KSp[slot * g.ld + r] = make_double2(0.0, 0.0);
      }
    }
  }
  double A[3][3];
  load_rr(g, b.top, A);
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n_add; e += gridDim.x * blockDim.x) {
    const int i = b.ext[e];
    double alfa = z[2 * i], r = z[2 * i + 1];
    const double Rl[4] = {R[4 * i], R[4 * i + 1], R[4 * i + 2], R[4 * i + 3]};
    const int l = 3 + 2 * (L + e);
    r = add_rn(r, add_rn(mul_rn(s_pose[0], cos(alfa)), mul_rn(s_pose[1], sin(alfa))));   /* :792 (Q8) */
    alfa = add_rn(alfa, s_pose[2]);                                                 /* :793 */
    double cw, sw;
    cos_sin(alfa, cw, sw);
    const double Gx[2][3] = {{0.0, 0.0, 1.0}, {cw, sw, 0.0}};
    const double Gl[2][2] = {{1.0, 0.0}, {sub_rn(mul_rn(s_y01[1], cw), mul_rn(s_y01[0], sw)), 1.0}};   /* :797-798 */
    normalize_radian(alfa);                                                       /* :801 */
    b.y[l] = alfa; b.y[l + 1] = r;
    b.ext_cs[2 * e] = cw; b.ext_cs[2 * e + 1] = sw;
    double GP[2][3] = {{0, 0, 0}, {0, 0, 0}};                                     /* :823 (NN) */
    for (int k = 0; k < 3; ++k)
      for (int ii = 0; ii < 2; ++ii) {
        const double t = mul_rn(1.0, Gx[ii][k]);
        if (t != 0.0) for (int jj = 0; jj < 3; ++jj) GP[ii][jj] = add_rn(GP[ii][jj], mul_rn(t, A[k][jj]));
      }
    double Pll[2][2];
    for (int ii = 0; ii < 2; ++ii)                                                /* :827 (NT) */
      for (int jj = 0; jj < 2; ++jj) {
        double t = 0.0;
        for (int k = 0; k < 3; ++k) t = add_rn(t, mul_rn(GP[ii][k], Gx[jj][k]));
        Pll[ii][jj] = add_rn(0.0, mul_rn(1.0, t));
      }
    double GR[2][2] = {{0, 0}, {0, 0}};                                           /* :831 (NN) */
    for (int k = 0; k < 2; ++k)
      for (int ii = 0; ii < 2; ++ii) {
        const double t = mul_rn(1.0, Gl[ii][k]);
        if (t != 0.0) for (int jj = 0; jj < 2; ++jj) GR[ii][jj] = add_rn(GR[ii][jj], mul_rn(t, Rl[k * 2 + jj]));
      }
    for (int ii = 0; ii < 2; ++ii)                                                /* :835, :839 */
      for (int jj = 0; jj < 2; ++jj) {
        double t = 0.0;
        for (int k = 0; k < 2; ++k) t = add_rn(t, mul_rn(GR[ii][k], Gl[jj][k]));
        Pll[ii][jj] = add_rn(Pll[ii][jj], add_rn(0.0, mul_rn(1.0, t)));
      }
    b.diag[4 * (L + e)] = Pll[0][0]; b.diag[4 * (L + e) + 1] = Pll[0][1]; b.diag[4 * (L + e) + 2] = Pll[1][1];
    b.diag[4 * (L + e) + 3] = 0.0;
    for (int k = 0; k < 3; ++k) {                                                 /* :856-860 for columns 0..2 */
      double r0 = 0.0, r1 = 0.0;
      for (int kk = 0; kk < 3; ++kk) {
        axpy_skip(r0, mul_rn(1.0, Gx[0][kk]), A[kk][k]);
        axpy_skip(r1, mul_rn(1.0, Gx[1][kk]), A[kk][k]);
      }
      b.top[(size_t)k * g.ld + l] = r0;
      b.top[(size_t)k * g.ld + l + 1] = r1;
    }
  }
  /* ++savedLineCount (Robot.cpp:866) for every appended line, then the reset test (:893-904).  Done here, by the one block of
   * this kernel, instead of in a third launch after phase B: phase B takes the line count from before the append (L0). */
  __syncthreads();
  if (threadIdx.x == 0) {
    st->L0 = L;
    int Ln = L + n_add;
    const bool reset = Ln > g.cap - g.headroom;
    if (reset) { Ln = 0; st->resets += 1; }
    st->L = Ln;
    /* what this scan's sweep will need.  A reset voids the pending terms (they describe the old map): a scan that continues
     * the sweep group carries none of them, and the group's sweep folds only terms formed after the reset. */
    if (view) { view->cnt = reset ? 0 : b.pidx[m] - st->pbase; view->L = Ln; }
  }
}

/* Robot.cpp:856-860 phase B: the new landmarks' column blocks P[k, l..l+1] = Gx * P[0:3, k], 3 <= k < l.
 * Threads run along the new columns (coalesced row writes); blockIdx.y strides over the rows. */
/* P2 != NULL: the new columns go into that buffer too -- the covariance the next scan of an open sweep group reads
 * (DESIGN section 5); there they are dead columns of the sweep in flight, which reads that buffer. */
__global__ void __launch_bounds__(EKF_BLOCK) k_end_scan_b(EkfGeom g, EkfBuffers b, double* __restrict__ P2) {
  const EkfDevState* st = b.st;
  const int n_add = st->n_added;
  const int L = st->L0;                                        /* lines before this scan's append (k_end_scan_a) */
  const int c_idx = blockIdx.x * blockDim.x + threadIdx.x;     /* 0 .. 2*n_add-1 */
  if (c_idx >= 2 * n_add) return;
  const int e = c_idx >> 1, tsel = c_idx & 1;
  const int l = 3 + 2 * (L + e);
  const int col = l + tsel;
  const double cw = b.ext_cs[2 * e], sw = b.ext_cs[2 * e + 1];
  const double* t0p = b.top; const double* t1p = b.top + g.ld; const double* t2p = b.top + 2 * (size_t)g.ld;
  for (int k = 3 + blockIdx.y; k < l; k += gridDim.y) {
    if (g.world > 1 && owner_of_row(g, k) != g.rank) continue;
    double v;
    if (tsel == 0) { v = 0.0; axpy_skip(v, 1.0, t2p[k]); }
    else { v = 0.0; axpy_skip(v, cw, t0p[k]); axpy_skip(v, sw, t1p[k]); }
    b.P[local_row(g, k) * g.ld + col] = v;
    if (P2) P2[local_row(g, k) * g.ld + col] = v;
  }
}

/* ------------------------------------------------------------------------------------------------ */
/* symmetrised read-out of rows [r0, r0+nr) x cols [c0, c0+nc) (zeros outside the live part).  In the
 * sharded mode each rank emits only what it owns (hot elements: rank 0), so the ranks' outputs sum to
 * the full matrix. */
__global__ void __launch_bounds__(EKF_BLOCK) k_assemble(EkfGeom g, EkfBuffers b, int r0, int nr, int c0, int nc,
                                                        double* __restrict__ out, int ld_out) {
  const int nl = 3 + 2 * b.st->L;
  const long long total = (long long)nr * nc;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
       t += (long long)gridDim.x * blockDim.x) {
    const int r = r0 + (int)(t / nc), q = c0 + (int)(t % nc);
    double v = 0.0;
    if (r < nl && q < nl) {
      const int lo = min(r, q), hi = max(r, q);
      if (is_hot(lo, hi)) { if (g.rank == 0) v = hot_value(g, b, lo, hi); }
      else if (g.world == 1 || owner_of_row(g, lo) == g.rank) v = b.P[local_row(g, lo) * g.ld + hi];
    }
    out[(size_t)(r - r0) * ld_out + (q - c0)] = v;
  }
}

/* inverse of k_assemble for ekf_upload: rows [r0, r0+nr) of a full row-major matrix (stride ld_in) */
__global__ void __launch_bounds__(EKF_BLOCK) k_scatter(EkfGeom g, EkfBuffers b, int r0, int nr, int nl,
                                                       const double* __restrict__ in, int ld_in) {
  const long long total = (long long)nr * nl;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total;
       t += (long long)gridDim.x * blockDim.x) {
    const int r = r0 + (int)(t / nl), q = (int)(t % nl);
    if (q < r) continue;                       /* upper triangle is authoritative */
    const double v = in[(size_t)(r - r0) * ld_in + q];
    if (r <= 2) b.top[(size_t)r * g.ld + q] = v;
    else if (is_hot(r, q)) {
      const int j = (r - 3) >> 1;
      if (r & 1) b.diag[4 * j + (q - r)] = v; else b.diag[4 * j + 2] = v;
    } else if (g.world == 1 || owner_of_row(g, r) == g.rank) b.P[local_row(g, r) * g.ld + q] = v;
  }
}

/* trace / sum / sum of squares of the symmetrised live covariance.  One block per row, fixed-order
 * tree inside the block, then a single block folds the per-row partials in index order. */
__global__ void __launch_bounds__(EKF_BLOCK) k_cov_rows(EkfGeom g, EkfBuffers b, double* __restrict__ partials) {
  __shared__ double s_sum[EKF_BLOCK], s_sq[EKF_BLOCK];
  const int nl = 3 + 2 * b.st->L;
  for (int r = blockIdx.x; r < nl; r += gridDim.x) {
    double sum = 0.0, sq = 0.0;
    for (int q = threadIdx.x; q < nl; q += blockDim.x) {
      const int lo = min(r, q), hi = max(r, q);
      double v = 0.0;
      if (is_hot(lo, hi)) { if (g.rank == 0) v = hot_value(g, b, lo, hi); }
      else if (g.world == 1 || owner_of_row(g, lo) == g.rank) v = b.P[local_row(g, lo) * g.ld + hi];
      sum += v; sq += v * v;
    }
    s_sum[threadIdx.x] = sum; s_sq[threadIdx.x] = sq;
    __syncthreads();
    for (int w = EKF_BLOCK / 2; w > 0; w >>= 1) {
      if (threadIdx.x < w) { s_sum[threadIdx.x] += s_sum[threadIdx.x + w]; s_sq[threadIdx.x] += s_sq[threadIdx.x + w]; }
      __syncthreads();
    }
    if (threadIdx.x == 0) {
      partials[3 * (size_t)r] = (g.rank == 0) ? hot_value(g, b, r, r) : 0.0;
      partials[3 * (size_t)r + 1] = s_sum[0];
      partials[3 * (size_t)r + 2] = s_sq[0];
    }
    __syncthreads();
  }
}
__global__ void k_cov_fold(EkfBuffers b, const double* __restrict__ partials, double* __restrict__ out3) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const int nl = 3 + 2 * b.st->L;
    double tr = 0.0, sum = 0.0, sq = 0.0;
    for (int r = 0; r < nl; ++r) { tr += partials[3 * (size_t)r]; sum += partials[3 * (size_t)r + 1]; sq += partials[3 * (size_t)r + 2]; }
    out3[0] = tr; out3[1] = sum; out3[2] = sq;
  }
}

/* roofline probe: m zero-valued pending terms (P is unchanged bit for bit by the sweep) */
__global__ void k_zero_pending(EkfGeom g, EkfBuffers b, int m, int* np) {
  const size_t total = (size_t)m * g.ld;
  for (size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    b.Kp[t] = make_double2(0.0, 0.0); b.KSp[t] = make_double2(0.0, 0.0);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) *np = m;
}

/* ------------------------------------------------------------------------------------------------ */
/* Landmark removal (ekf_remove_lines, DESIGN section 3): pure data movement.  keep[i] = old state index of new state
 * index i (i < nl, strictly increasing, keep[i] = i for i < 3). */

/* Hot storage: y, rows 0..2 of `top` and the 2x2 diagonal blocks of the kept landmarks.  put = 0 gathers them into
 * stage = [y (nl) | top rows (3 x nl) | diag (4 x L)]; put = 1 copies the stage back in place (the two launches are the
 * ordering: a kept entry's source may be another kept entry's destination). */
__global__ void __launch_bounds__(EKF_BLOCK) k_remove_hot(EkfGeom g, EkfBuffers b, const int* __restrict__ keep, int nl,
                                                          double* __restrict__ stage, int put) {
  const long long total = 4LL * nl + 2LL * (nl - 3);
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    double* dst;
    const double* src;
    if (t < nl) { dst = b.y + t; src = b.y + keep[t]; }
    else if (t < 4LL * nl) {
      const int k = (int)((t - nl) / nl), c = (int)((t - nl) % nl);
      dst = b.top + (size_t)k * g.ld + c; src = b.top + (size_t)k * g.ld + keep[c];
    } else {
      const int e = (int)(t - 4LL * nl), j = e >> 2, w = e & 3;
      dst = b.diag + 4 * j + w; src = b.diag + 4 * ((keep[3 + 2 * j] - 3) >> 1) + w;
    }
    if (put) *dst = stage[t]; else stage[t] = *src;
  }
}

/* Cold covariance, rows [r0, r0 + nr) of the compacted live upper triangle.  Destination row r (at dst + (r - dst_row0) *
 * ld_dst) gets, in columns max(r, c_from) .. nl-1, the source elements (keep[r], keep[c]) (GATHER) or (r, c) (the copy back
 * from the stage), source row i at src + (i - src_row0) * ld_src.  keep is increasing, so an upper destination element
 * has an upper source.  The kept runs between removed landmarks make each row's reads piecewise contiguous: one CTA per
 * row, RM_UNROLL independent 8-byte loads in flight per thread, read-once data streamed past L1/L2 (ld.cs / st.cs). */
#define RM_UNROLL 4
template <bool GATHER>
__global__ void __launch_bounds__(EKF_BLOCK) k_remove_cold(const double* __restrict__ src, size_t ld_src, int src_row0,
                                                           double* __restrict__ dst, size_t ld_dst, int dst_row0,
                                                           const int* __restrict__ keep, int r0, int nr, int nl, int c_from) {
  for (int i = blockIdx.x; i < nr; i += gridDim.x) {
    const int r = r0 + i;
    const double* s = src + (size_t)((GATHER ? __ldg(keep + r) : r) - src_row0) * ld_src;
    double* d = dst + (size_t)(r - dst_row0) * ld_dst;
    for (int c = max(r, c_from) + threadIdx.x; c < nl; c += RM_UNROLL * EKF_BLOCK) {
      double v[RM_UNROLL];
#pragma unroll
      for (int u = 0; u < RM_UNROLL; ++u) {
        const int cc = c + u * EKF_BLOCK;
        if (cc < nl) v[u] = __ldcs(s + (GATHER ? __ldg(keep + cc) : cc));
      }
#pragma unroll
      for (int u = 0; u < RM_UNROLL; ++u) {
        const int cc = c + u * EKF_BLOCK;
        if (cc < nl) __stcs(d + cc, v[u]);
      }
    }
  }
}

/* ------------------------------------------------------------------------------------------------ */
/* Landmark insertion (ekf_insert_lines, DESIGN section 3.3): y' = [y, lines], P' = [[P, 0], [0, C]], pure data movement.
 * The new landmarks are j = L .. L+k-1, state indices nl_old .. nl-1 (nl_old = 3 + 2 L, nl = nl_old + 2 k). */

/* Hot storage.  src[5 e .. 5 e + 5) = (alfa, r, C[a,a], C[a,b], C[b,b]) of new landmark e: its y entries (alfa wrapped
 * as the augmentation wraps it, Robot.cpp:801), its zero columns of `top` and its 2x2 diagonal block (pad 0, as
 * k_end_scan_a writes it). */
__global__ void __launch_bounds__(EKF_BLOCK) k_insert_hot(EkfGeom g, EkfBuffers b, int L, int k,
                                                          const double* __restrict__ src) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < k; e += gridDim.x * blockDim.x) {
    const double* s = src + 5 * e;
    const int a = 3 + 2 * (L + e);
    double alfa = s[0];
    normalize_radian(alfa);
    b.y[a] = alfa; b.y[a + 1] = s[1];
    for (int q = 0; q < 3; ++q) { b.top[(size_t)q * g.ld + a] = 0.0; b.top[(size_t)q * g.ld + a + 1] = 0.0; }
    double* dg = b.diag + 4 * (size_t)(L + e);
    dg[0] = s[2]; dg[1] = s[3]; dg[2] = s[4]; dg[3] = 0.0;
  }
}

/* Cold covariance, rows [r0, r0 + nr) of the live upper triangle, columns max(r, nl_old) .. nl-1 (the new columns).  A row
 * above the new block (r < nl_old) gets zeros; a new row gets row r - nl_old of the new block C (2k wide, row i of it at
 * blk + (i - blk_row0) * 2k), or zeros when blk = NULL.  One CTA per row: a scalar store up to the first 16-byte boundary,
 * then double2 streaming stores along the row (rows start on 2 KB boundaries, so even columns are 16-byte aligned). */
__global__ void __launch_bounds__(EKF_BLOCK) k_insert_cold(double* __restrict__ P, size_t ld, int nl_old, int nl, int r0,
                                                           int nr, const double* __restrict__ blk, int blk_row0) {
  const int w = nl - nl_old;
  for (int i = blockIdx.x; i < nr; i += gridDim.x) {
    const int r = r0 + i;
    const int c0 = max(r, nl_old);
    double* d = P + (size_t)r * ld;
    const double* s = (blk && r >= nl_old) ? blk + (size_t)(r - nl_old - blk_row0) * w - nl_old : 0;
    int c = c0;
    if (c & 1) { if (threadIdx.x == 0) __stcs(d + c, s ? __ldg(s + c) : 0.0); ++c; }
    for (int q = c + 2 * threadIdx.x; q < nl; q += 2 * EKF_BLOCK) {
      if (q + 1 < nl) __stcs(reinterpret_cast<double2*>(d + q), s ? make_double2(__ldg(s + q), __ldg(s + q + 1)) : make_double2(0.0, 0.0));
      else __stcs(d + q, s ? __ldg(s + q) : 0.0);
    }
  }
}

/* ------------------------------------------------------------------------------------------------ */
/* Absolute pose fix (ekf_observe_pose, DESIGN section 3.2).  H = the D selected rows of [I_3 0], so P H' is D columns of
 * P among 0..2 -- all in `top`, hot and always current -- and H P H' is a D x D block of the robot rows.  The arithmetic is
 * the reference-BLAS pattern of Robot.cpp:516-602 with D x D blocks: PHt = P H', S = H P H' + R, S^-1 by LU, d2 = v' S^-1 v
 * (TN then NN as at :479-483), K = PHt S^-1 and KS = K S (NN), P -= KS K' as two rank-2 terms, y += K v, then the wrap
 * of y[2] and the pose mirrors (:596-602).  Products with the structural 0 / 1 entries of H are exact and not issued. */
struct PoseGate { double S[9], Si[9], v[3], d2; int status; };

template <int D>
__device__ __forceinline__ void pose_gate(const EkfGeom& g, const EkfBuffers& b, const EkfPoseFix& f, PoseGate& G) {
#pragma unroll
  for (int i = 0; i < D; ++i)
#pragma unroll
    for (int k = 0; k < D; ++k) {                                     /* upper triangle of the robot block, plus R_sel */
      const int r = min(f.sel[i], f.sel[k]), c = max(f.sel[i], f.sel[k]);
      G.S[3 * i + k] = add_rn(b.top[(size_t)r * g.ld + c], f.R[3 * i + k]);
    }
  const int sing = invDxD_lu<D>(G.S, G.Si);
#pragma unroll
  for (int i = 0; i < D; ++i) {
    double v = sub_rn(f.z[i], b.y[f.sel[i]]);
    if (f.sel[i] == 2) normalize_radian(v);
    G.v[i] = v;
  }
  double w[D];                                                        /* v' S^-1 (TN) */
#pragma unroll
  for (int c = 0; c < D; ++c) w[c] = 0.0;
#pragma unroll
  for (int k = 0; k < D; ++k)
#pragma unroll
    for (int c = 0; c < D; ++c) axpy_skip(w[c], G.v[k], G.Si[3 * k + c]);
  double d2 = 0.0;                                                    /* (v' S^-1) v (NN) */
#pragma unroll
  for (int c = 0; c < D; ++c) axpy_skip(d2, w[c], G.v[c]);
  G.d2 = d2;
  /* accepted iff S is nonsingular and d2 <= d2max (false for a NaN d2) */
  G.status = sing ? EKF_FIX_SINGULAR : (d2 <= f.d2max ? EKF_FIX_ACCEPTED : EKF_FIX_REJECTED);
}

/* Every block forms the gate redundantly (a few hundred flops); block 0 publishes it.  Each thread then writes the gain
 * rows of its state indices as term 1 (slot 0) and, for D = 3, term 2 (K2, KS2). */
template <int D>
__global__ void __launch_bounds__(EKF_BLOCK) k_pose_gain(EkfGeom g, EkfBuffers b, EkfPoseFix f, double2* __restrict__ K2,
                                                         double2* __restrict__ KS2) {
  __shared__ PoseGate sG;
  EkfDevState* st = b.st;
  if (threadIdx.x == 0) {
    pose_gate<D>(g, b, f, sG);
    if (blockIdx.x == 0) {
      st->fix_status = sG.status;
      for (int t = 0; t < 9; ++t) st->fix_S[t] = (t / 3 < D && t % 3 < D) ? sG.S[t] : 0.0;
      for (int t = 0; t < 3; ++t) st->fix_v[t] = t < D ? sG.v[t] : 0.0;
      st->fix_d2 = sG.d2;
    }
  }
  __syncthreads();
  if (sG.status != EKF_FIX_ACCEPTED) return;
  const int nl = 3 + 2 * st->L;
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < nl; r += gridDim.x * blockDim.x) {
    double ph[D];                                                     /* P H': P[r, sel[i]] through the upper storage */
#pragma unroll
    for (int i = 0; i < D; ++i) ph[i] = b.top[(size_t)min(r, f.sel[i]) * g.ld + max(r, f.sel[i])];
    double k[D], ks[D];
#pragma unroll
    for (int c = 0; c < D; ++c) { k[c] = 0.0; ks[c] = 0.0; }
#pragma unroll
    for (int i = 0; i < D; ++i)                                       /* K = PHt S^-1 (NN) */
#pragma unroll
      for (int c = 0; c < D; ++c) axpy_skip(k[c], ph[i], sG.Si[3 * i + c]);
#pragma unroll
    for (int i = 0; i < D; ++i)                                       /* K S (NN) */
#pragma unroll
      for (int c = 0; c < D; ++c) axpy_skip(ks[c], k[i], sG.S[3 * i + c]);
    b.Kp[r] = make_double2(k[0], D > 1 ? k[1] : 0.0);
    b.KSp[r] = make_double2(ks[0], D > 1 ? ks[1] : 0.0);
    if (D == 3) { K2[r] = make_double2(k[D - 1], 0.0); KS2[r] = make_double2(ks[D - 1], 0.0); }
  }
}

/* P -= KS K' on the hot elements (rows 0..2, the 2x2 diagonal blocks), term 1 then term 2 as the sweep folds them into the
 * cold ones; y += K v; the wrap of y[2]; pose and x_pre follow y[0:3] (Robot.cpp:596-602). */
template <int D>
__global__ void __launch_bounds__(EKF_BLOCK) k_pose_apply(EkfGeom g, EkfBuffers b, const double2* __restrict__ K2,
                                                          const double2* __restrict__ KS2, int max_np) {
  EkfDevState* st = b.st;
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  if (st->fix_status != EKF_FIX_ACCEPTED) {
    if (gid == 0) st->np = 0;                                         /* nothing for the sweep: P stays bit for bit */
    return;
  }
  const int nl = 3 + 2 * st->L;
  const double v0 = st->fix_v[0], v1 = st->fix_v[1], v2 = st->fix_v[2];
  const double2* K = b.Kp;
  const double2* KS = b.KSp;
  const double2 z2 = make_double2(0.0, 0.0);
  double2 ks1[3], ks2[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) { ks1[r] = KS[r]; ks2[r] = D == 3 ? KS2[r] : z2; }
  for (int q = 3 + gid; q < nl; q += gridDim.x * blockDim.x) {
    const double2 k1 = K[q], k2 = D == 3 ? K2[q] : z2;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      double p = sub_rank2(b.top[(size_t)r * g.ld + q], ks1[r], k1);
      if (D == 3) p = sub_rank2(p, ks2[r], k2);
      b.top[(size_t)r * g.ld + q] = p;
    }
    const double2 s1 = KS[q], s2 = D == 3 ? KS2[q] : z2;
    const int jj = (q - 3) >> 1;
    if (q & 1) {                                                      /* q = a: (a,a), (a,b) */
      const double2 k1b = K[q + 1], k2b = D == 3 ? K2[q + 1] : z2;
      double paa = sub_rank2(b.diag[4 * jj], s1, k1), pab = sub_rank2(b.diag[4 * jj + 1], s1, k1b);
      if (D == 3) { paa = sub_rank2(paa, s2, k2); pab = sub_rank2(pab, s2, k2b); }
      b.diag[4 * jj] = paa; b.diag[4 * jj + 1] = pab;
    } else {                                                          /* q = b: (b,b) */
      double pbb = sub_rank2(b.diag[4 * jj + 2], s1, k1);
      if (D == 3) pbb = sub_rank2(pbb, s2, k2);
      b.diag[4 * jj + 2] = pbb;
    }
    double t = 0.0;                                                   /* y += K v (NN) */
    axpy_skip(t, k1.x, v0);
    if (D > 1) axpy_skip(t, k1.y, v1);
    if (D > 2) axpy_skip(t, k2.x, v2);
    b.y[q] = add_rn(b.y[q], t);
  }
  if (gid == 0) {
    const double2 kk1[3] = {K[0], K[1], K[2]};
    const double2 kk2[3] = {D == 3 ? K2[0] : z2, D == 3 ? K2[1] : z2, D == 3 ? K2[2] : z2};
    for (int r = 0; r < 3; ++r)
      for (int q = r; q < 3; ++q) {
        double p = sub_rank2(b.top[(size_t)r * g.ld + q], ks1[r], kk1[q]);
        if (D == 3) p = sub_rank2(p, ks2[r], kk2[q]);
        b.top[(size_t)r * g.ld + q] = p;
      }
    double yn[3];
    for (int r = 0; r < 3; ++r) {
      double t = 0.0;
      axpy_skip(t, kk1[r].x, v0);
      if (D > 1) axpy_skip(t, kk1[r].y, v1);
      if (D > 2) axpy_skip(t, kk2[r].x, v2);
      yn[r] = add_rn(b.y[r], t);
    }
    normalize_radian(yn[2]);
    for (int r = 0; r < 3; ++r) { b.y[r] = yn[r]; st->pose[r] = yn[r]; st->x_pre[r] = yn[r]; }
    st->np = min(max_np, D == 3 ? 2 : 1);
  }
}

/* one pending slot only: term 2 moves into slot 0 for a second one-term sweep */
__global__ void __launch_bounds__(EKF_BLOCK) k_pose_term2(EkfGeom g, EkfBuffers b, int d, const double2* __restrict__ K2,
                                                          const double2* __restrict__ KS2) {
  const bool on = d == 3 && b.st->fix_status == EKF_FIX_ACCEPTED;
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  if (gid == 0) b.st->np = on ? 1 : 0;
  if (!on) return;
  const int nl = 3 + 2 * b.st->L;
  for (int r = gid; r < nl; r += gridDim.x * blockDim.x) { b.Kp[r] = K2[r]; b.KSp[r] = KS2[r]; }
}

inline int blocks_for(long long n, int cap = 1 << 20) {
  long long bl = (n + EKF_BLOCK - 1) / EKF_BLOCK;
  if (bl < 1) bl = 1;
  if (bl > cap) bl = cap;
  return (int)bl;
}

}  // namespace

/* ---------------------------------------- launchers ---------------------------------------------- */
cudaError_t ekf_launch_init(const EkfGeom& g, const EkfBuffers& b, cudaStream_t s) {
  k_init<<<1, 32, 0, s>>>(g, b);
  return cudaGetLastError();
}
cudaError_t ekf_launch_predict(const EkfGeom& g, const EkfBuffers& b, const double* d_u, const double* d_x_t0,
                               int m, int L_ub, cudaStream_t s, const int* carry) {
  const int work = (3 + 2 * L_ub > m) ? 3 + 2 * L_ub : m;
  k_predict<<<blocks_for(work, 1024), EKF_BLOCK, 0, s>>>(g, b, d_u, d_x_t0, m, carry);
  return cudaGetLastError();
}
cudaError_t ekf_launch_associate(const EkfGeom& g, const EkfBuffers& b, const double* d_z, const double* d_R,
                                 int line, int L_ub, cudaStream_t s) {
  if (L_ub <= 0) return cudaSuccess;
  k_associate<<<blocks_for(L_ub), EKF_BLOCK, 0, s>>>(g, b, d_z, d_R, line);
  return cudaGetLastError();
}
cudaError_t ekf_launch_gain(const EkfGeom& g, const EkfBuffers& b, const double* d_z, const double* d_R,
                            int line, int j_override, int mode, int L_ub, int max_batch, cudaStream_t s) {
  if (L_ub <= 0) return cudaSuccess;
  k_gain<<<blocks_for(3 + 2 * L_ub, 2048), EKF_BLOCK, 0, s>>>(g, b, d_z, d_R, line, j_override, mode, max_batch);
  return cudaGetLastError();
}
cudaError_t ekf_launch_apply(const EkfGeom& g, const EkfBuffers& b, int line, int j_override, int L_ub,
                             cudaStream_t s) {
  k_apply<<<blocks_for(3 + 2 * L_ub, 2048), EKF_BLOCK, 0, s>>>(g, b, line, j_override);
  return cudaGetLastError();
}
/* largest cluster (16, else 8) the device can co-schedule for the line-loop kernel */
#ifdef EKF_LINE_TIMING
extern "C" int ekf_debug_line_timing(unsigned long long* out, int n) {
  return (int)cudaMemcpyFromSymbol(out, g_line_ts, sizeof(unsigned long long) * (size_t)n);
}
#endif
/* Kernels of the line stream must be able to share an SM with a resident sweep CTA (which runs with the
 * maximum shared-memory carve-out): an SM cannot host kernels with different carve-outs at the same time. */
void ekf_prefer_max_smem_carveout(void) {
  const int c = cudaSharedmemCarveoutMaxShared;
  cudaFuncSetAttribute(k_predict, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  cudaFuncSetAttribute(k_scan_lines<512, true, false>, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  cudaFuncSetAttribute(k_scan_lines<512, true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  cudaFuncSetAttribute(k_scan_lines<512, false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  cudaFuncSetAttribute(k_scan_lines2<512, true, true>, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  cudaFuncSetAttribute(k_scan_lines2<512, true, false>, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  cudaFuncSetAttribute(k_scan_lines2<512, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  cudaFuncSetAttribute(k_scan_lines2<256, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  cudaFuncSetAttribute(k_scan_lines2<512, false, false>, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  cudaFuncSetAttribute(k_end_scan_a, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  cudaFuncSetAttribute(k_end_scan_b, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  cudaFuncSetAttribute(k_chunk_mark, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  cudaFuncSetAttribute(k_queue_all, cudaFuncAttributePreferredSharedMemoryCarveout, c);
  (void)cudaGetLastError();
}
/* EKF_LINE_LOOP=1 keeps the first, two-barrier form of the line loop on one GPU too (A/B measurement and bit checks) */
static int line_loop_v1() { static int v = -1; if (v < 0) { const char* e = getenv("EKF_LINE_LOOP"); v = (e && atoi(e) == 1) ? 1 : 0; } return v; }
int ekf_pick_cluster(void) {
  cudaFuncSetAttribute(k_scan_lines<512, false, false>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  cudaFuncSetAttribute(k_scan_lines2<512, false, true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  cudaFuncSetAttribute(k_scan_lines2<256, false, true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  cudaFuncSetAttribute(k_scan_lines2<512, false, false>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  { const char* e = getenv("EKF_CLUSTER"); const int v = e ? atoi(e) : 0; if (v == 1 || v == 2 || v == 4 || v == 8) return v; }   /* A/B measurements */
  const int tries[2] = {16, 8};
  for (int t = 0; t < 2; ++t) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(tries[t]); cfg.blockDim = dim3(512);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = tries[t]; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    int n = 0;
    int n2 = 0;
    if (cudaOccupancyMaxActiveClusters(&n, k_scan_lines<512, false, false>, &cfg) == cudaSuccess && n >= 1 &&
        cudaOccupancyMaxActiveClusters(&n2, k_scan_lines2<512, false, false>, &cfg) == cudaSuccess && n2 >= 1) return tries[t];
  }
  (void)cudaGetLastError();
  return 8;
}
/* whether ekf_launch_scan_lines can run the scan's prediction as the prologue of the line loop (the one-barrier form only) */
int ekf_scan_lines_fuses_predict(const EkfPeers* peers) { return !line_loop_v1() && !(peers && peers->world > 1); }
cudaError_t ekf_launch_scan_lines(const EkfGeom& g, const EkfBuffers& b, const double* d_z, const double* d_R,
                                  int line0, int line1, int ctas, int coop, int own_slot0, int prev_slot0,
                                  const int* prev_cnt_ptr, const EkfPeers* peers, int L_ub, cudaStream_t s,
                                  const double* pred_u, const double* pred_x, int pred_m, const int* pred_carry) {
  if (line1 <= line0) return cudaSuccess;
  if (pred_u && !ekf_scan_lines_fuses_predict(peers)) return cudaErrorInvalidValue;
  EkfPeers pe;
  memset(&pe, 0, sizeof pe);
  pe.world = 1;
  if (peers) pe = *peers;
  if (coop) {
    void* args[] = {(void*)&g, (void*)&b, (void*)&d_z, (void*)&d_R, (void*)&line0, (void*)&line1, (void*)&own_slot0,
                    (void*)&prev_slot0, (void*)&prev_cnt_ptr, (void*)&pe};
    if (peers && peers->world > 1)
      return cudaLaunchCooperativeKernel((const void*)k_scan_lines<512, true, true>, dim3(ctas), dim3(512), args, 0, s);
    if (line_loop_v1())
      return cudaLaunchCooperativeKernel((const void*)k_scan_lines<512, true, false>, dim3(ctas), dim3(512), args, 0, s);
    void* args2[] = {(void*)&g, (void*)&b, (void*)&d_z, (void*)&d_R, (void*)&line0, (void*)&line1, (void*)&own_slot0,
                     (void*)&prev_slot0, (void*)&prev_cnt_ptr, (void*)&pred_u, (void*)&pred_x, (void*)&pred_m, (void*)&pred_carry};
    /* 256-thread CTAs (EKF_LINE_THREADS=256, twice the SMs for the same map): up to 255 registers per thread -- none of the
     * line loop's state spills */
    static int lt = -1;
    if (lt < 0) { const char* e = getenv("EKF_LINE_THREADS"); lt = e ? atoi(e) : 0; }
    if (L_ub > g.cap) L_ub = g.cap;
    if (lt == 256 && L_ub <= ctas * 256)
      return cudaLaunchCooperativeKernel((const void*)k_scan_lines2<256, true, true>, dim3(ctas), dim3(256), args2, 0, s);
    /* at most one landmark per thread (host-side bound): the form that keeps the hot entries in registers */
    if (L_ub <= ctas * 512) return cudaLaunchCooperativeKernel((const void*)k_scan_lines2<512, true, true>, dim3(ctas), dim3(512), args2, 0, s);
    return cudaLaunchCooperativeKernel((const void*)k_scan_lines2<512, true, false>, dim3(ctas), dim3(512), args2, 0, s);
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = dim3(ctas); cfg.blockDim = dim3(512); cfg.dynamicSmemBytes = 0; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = ctas; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  if (line_loop_v1())
    return cudaLaunchKernelEx(&cfg, k_scan_lines<512, false, false>, g, b, d_z, d_R, line0, line1, own_slot0, prev_slot0, prev_cnt_ptr, pe);
  if (L_ub <= ctas * 256) {
    /* small maps: 256-thread CTAs may use up to 255 registers -- no spills on the per-line critical path */
    cfg.blockDim = dim3(256);
    return cudaLaunchKernelEx(&cfg, k_scan_lines2<256, false, true>, g, b, d_z, d_R, line0, line1, own_slot0, prev_slot0, prev_cnt_ptr, pred_u, pred_x, pred_m, pred_carry);
  }
  if (L_ub <= ctas * 512)
    return cudaLaunchKernelEx(&cfg, k_scan_lines2<512, false, true>, g, b, d_z, d_R, line0, line1, own_slot0, prev_slot0, prev_cnt_ptr, pred_u, pred_x, pred_m, pred_carry);
  return cudaLaunchKernelEx(&cfg, k_scan_lines2<512, false, false>, g, b, d_z, d_R, line0, line1, own_slot0, prev_slot0, prev_cnt_ptr, pred_u, pred_x, pred_m, pred_carry);
}
cudaError_t ekf_launch_flush_done(const EkfBuffers& b, int next_line, cudaStream_t s) {
  k_flush_done<<<1, 32, 0, s>>>(b, next_line);
  return cudaGetLastError();
}
cudaError_t ekf_launch_chunk_mark(const EkfBuffers& b, int next_line, EkfScanView* view, cudaStream_t s) {
  k_chunk_mark<<<1, 32, 0, s>>>(b, next_line, view);
  return cudaGetLastError();
}
cudaError_t ekf_launch_queue_all(const EkfGeom& g, const EkfBuffers& b, int m, cudaStream_t s) {
  if (m <= 0) return cudaSuccess;
  k_queue_all<<<blocks_for(m, 1024), EKF_BLOCK, 0, s>>>(g, b, m);
  return cudaGetLastError();
}
int ekf_sweep_grid_ub(const EkfGeom& g, int L_ub) {
  const int nl = 3 + 2 * L_ub;
  const int T = (nl + EKF_TILE - 1) / EKF_TILE;
  if (g.rank >= T) return 0;
  const long long K = (T - g.rank + g.world - 1) / g.world;
  const long long total = K * (long long)(T - g.rank) - (long long)g.world * K * (K - 1) / 2;
  return (int)total;
}
cudaError_t ekf_launch_sweep(const EkfGeom& g, const EkfBuffers& b, const int* np_ptr, int np_ub, int L_ub,
                             cudaStream_t s) {
  const int grid = ekf_sweep_grid_ub(g, L_ub);
  if (grid <= 0 || np_ub <= 0) return cudaSuccess;
  if (np_ub <= 1) k_sweep<1><<<grid, EKF_BLOCK, 0, s>>>(g, b, np_ptr);
  else if (np_ub <= 2) k_sweep<2><<<grid, EKF_BLOCK, 0, s>>>(g, b, np_ptr);
  else if (np_ub <= 4) k_sweep<4><<<grid, EKF_BLOCK, 0, s>>>(g, b, np_ptr);
  else k_sweep<8><<<grid, EKF_BLOCK, 0, s>>>(g, b, np_ptr);
  return cudaGetLastError();
}
template <int TR, int TC, int STAGES, int CW, int C>
static cudaError_t launch_sweep_shape(const EkfGeom& g, const EkfBuffers& b, const CUtensorMap* m, const CUtensorMap* mK,
                                      const CUtensorMap* mKS, double* dst, int slot0,
                                      const EkfScanView* view, unsigned long long* counters, int np_ub, int grid, cudaStream_t s,
                                      const CUtensorMap* m_dst = 0) {
  const size_t smem = sizeof(SweepShared<TR, TC, STAGES, C>) + 1024;
  static bool attr_set[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(k_sweep_pipe<TR, TC, STAGES, CW, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  if (counters) {   /* one tile counter per pass */
    cudaError_t e = cudaMemsetAsync(counters, 0, sizeof(unsigned long long) * ((np_ub + C - 1) / C), s);
    if (e != cudaSuccess) return e;
  }
  for (int c0 = 0; c0 < np_ub; c0 += C) {
    /* an out-of-place sweep of more than C terms: the first pass goes source -> destination, the others fold the rest in
     * place on the destination (m_dst = its tensor map) */
    EkfBuffers bb = b;
    if (c0 > 0 && dst != b.P) { bb.P = dst; m = m_dst; }
    k_sweep_pipe<TR, TC, STAGES, CW, C><<<grid, (CW + 1) * 32, smem, s>>>(g, bb, *m, *mK, *mKS, dst, c0, slot0, view, counters ? counters + c0 / C : 0);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
template <int STAGES, int C>
static cudaError_t launch_sweep_quad(const EkfGeom& g, const EkfBuffers& b, const CUtensorMap* m, const CUtensorMap* mK,
                                     const CUtensorMap* mKS, double* dst, int slot0,
                                     const EkfScanView* view, unsigned long long* counters, int np_ub, int grid, cudaStream_t s,
                                     const CUtensorMap* m_dst = 0) {
  const size_t smem = sizeof(SweepShared<64, 64, STAGES, C>) + 1024;
  static bool attr_set[64] = {false};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(k_sweep_quad<STAGES, C>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  if (counters) {   /* one tile counter per pass */
    cudaError_t e = cudaMemsetAsync(counters, 0, sizeof(unsigned long long) * ((np_ub + C - 1) / C), s);
    if (e != cudaSuccess) return e;
  }
  for (int c0 = 0; c0 < np_ub; c0 += C) {
    EkfBuffers bb = b;
    if (c0 > 0 && dst != b.P) { bb.P = dst; m = m_dst; }
    k_sweep_quad<STAGES, C><<<grid, 9 * 32, smem, s>>>(g, bb, *m, *mK, *mKS, dst, c0, slot0, view, counters ? counters + c0 / C : 0);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
template <int STAGES, int C>
static cudaError_t launch_sweep_dmma(const EkfGeom& g, const EkfBuffers& b, const CUtensorMap* m, const CUtensorMap* mK,
                                     const CUtensorMap* mKS, double* dst, int slot0,
                                     const EkfScanView* view, unsigned long long* counters, int np_ub, int grid, cudaStream_t s,
                                     const CUtensorMap* m_dst = 0) {
  const size_t smem = sizeof(SweepShared<64, 64, STAGES, C>) + 1024;
  static bool attr_set[64] = {false};
  /* EKF_DMMA_SPLIT=0: the stage is refilled in one step (A/B against the split refill) */
  static int split = -1;
  if (split < 0) { const char* e = getenv("EKF_DMMA_SPLIT"); split = (e && atoi(e) == 0) ? 0 : 1; }
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    cudaError_t e = cudaFuncSetAttribute(k_sweep_dmma<STAGES, C, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_sweep_dmma<STAGES, C, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  if (counters) {   /* one tile counter per pass */
    cudaError_t e = cudaMemsetAsync(counters, 0, sizeof(unsigned long long) * ((np_ub + C - 1) / C), s);
    if (e != cudaSuccess) return e;
  }
  for (int c0 = 0; c0 < np_ub; c0 += C) {
    EkfBuffers bb = b;
    if (c0 > 0 && dst != b.P) { bb.P = dst; m = m_dst; }
    if (split) k_sweep_dmma<STAGES, C, true><<<grid, 9 * 32, smem, s>>>(g, bb, *m, *mK, *mKS, dst, c0, slot0, view, counters ? counters + c0 / C : 0);
    else k_sweep_dmma<STAGES, C, false><<<grid, 9 * 32, smem, s>>>(g, bb, *m, *mK, *mKS, dst, c0, slot0, view, counters ? counters + c0 / C : 0);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
/* box of the TMA map of P: the tile itself, except for the tensor-core sweep (shape 10: eight 64 x 8 boxes per tile) */
void ekf_sweep_pbox(int shape, int* rows, int* cols) {
  if (shape == 10) { *rows = 64; *cols = 8; return; }
  ekf_sweep_shape(shape == 11 ? 0 : shape, rows, cols);
}
void ekf_sweep_shape(int shape, int* tr, int* tc) {
  switch (shape) { case 1: case 5: *tr = 32; *tc = 128; break; case 2: *tr = 16; *tc = 256; break; default: *tr = 64; *tc = 64; }
}
/* terms one pass of the sweep folds for a scan with np_ub pending terms */
int ekf_sweep_terms_per_pass(int shape, int np_ub) {
  if (shape != 0 && shape != 9 && shape != 10 && shape != 11) return SW_C;
  static int cap = -1;
  if (cap < 0) { const char* e = getenv("EKF_SWEEP_MAXC"); cap = e ? atoi(e) : 32; if (cap != 8 && cap != 16 && cap != 32) cap = 32; }
  const int want = np_ub <= 8 ? 8 : (np_ub <= 16 ? 16 : 32);
  return want < cap ? want : cap;
}
cudaError_t ekf_launch_sweep_tma(const EkfGeom& g, const EkfBuffers& b, const void* tmap, const void* tmap8, const void* tmapK, const void* tmapKS,
                                 double* dst, int slot0,
                                 const EkfScanView* view, unsigned long long* counters, int shape, int np_ub, int L_ub,
                                 int num_sms, cudaStream_t s, const void* tmap_dst, const void* tmap8_dst) {
  const int tiles = ekf_sweep_grid_ub(g, L_ub);
  if (tiles <= 0 || np_ub <= 0) return cudaSuccess;
  const int C = ekf_sweep_terms_per_pass(shape, np_ub);
  /* out-of-place form with more terms than one pass folds: needs the destination's tensor maps for the in-place rest */
  if (dst != b.P && np_ub > C && !tmap_dst) return cudaErrorInvalidValue;
  const CUtensorMap* md = reinterpret_cast<const CUtensorMap*>(tmap_dst);
  const CUtensorMap* md8 = reinterpret_cast<const CUtensorMap*>(tmap8_dst);
  const int grid = tiles < num_sms ? tiles : num_sms;      /* num_sms: SMs this sweep may occupy */
  const CUtensorMap* m = reinterpret_cast<const CUtensorMap*>(tmap);
  const CUtensorMap* m8 = reinterpret_cast<const CUtensorMap*>(tmap8);
  const CUtensorMap* mK = reinterpret_cast<const CUtensorMap*>(tmapK);
  /* default (shape 0): up to 8 pending terms the pass is HBM-bound on the DFMA consumers (k_sweep_quad, 0.96 of the
   * measured peak inside a step); beyond, the fp64 tensor-core consumers take over (k_sweep_dmma: 1.04 ms against
   * 1.22 ms at 32 terms, 10k landmarks).  Shape 10 forces the tensor cores for every count, shape 11 never uses them. */
  if (shape == 11) shape = 0;
  else if (shape == 0 && np_ub > 8 && m8) shape = 10;
  const CUtensorMap* mKS = reinterpret_cast<const CUtensorMap*>(tmapKS);
  /* EKF_SWEEP_STAGES=2|3: a shallower ring (fewer bytes in flight per SM: lower loaded memory latency for the line loop beside
   * the sweep, at the price of less latency tolerance in the sweep) -- measurement knob */
  static int stg = -1;
  if (stg < 0) { const char* e = getenv("EKF_SWEEP_STAGES"); stg = e ? atoi(e) : 0; }
  if (stg == 2 || stg == 3) {
    if (shape == 10 && C == 16 && stg == 2) return launch_sweep_dmma<2, 16>(g, b, m8, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md8);
    if (shape == 0 && C == 8) {
      if (stg == 2) return launch_sweep_quad<2, 8>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);
      return launch_sweep_quad<3, 8>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);
    }
  }
  switch (shape) {       /* shape % 4: tile shape; shape / 4: 0 = 8 consumer warps, 1 = 16 */
    case 1: return launch_sweep_shape<32, 128, 4, 8, 8>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);
    case 2: return launch_sweep_shape<16, 256, 3, 8, 8>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);
    case 4: return launch_sweep_shape<64, 64, 4, 16, 8>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);
    case 5: return launch_sweep_shape<32, 128, 4, 16, 8>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);
    case 8: return launch_sweep_shape<64, 64, 3, 8, 8>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);   /* 148 KB: leaves room for a co-resident line-loop CTA */
    case 10:       /* fp64 tensor cores (k_sweep_dmma) */
      if (!m8) return cudaErrorInvalidValue;
      if (dst != b.P && np_ub > C && !md8) return cudaErrorInvalidValue;
      if (C == 32) return launch_sweep_dmma<2, 32>(g, b, m8, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md8);
      if (C == 16) return launch_sweep_dmma<3, 16>(g, b, m8, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md8);
      return launch_sweep_dmma<4, 8>(g, b, m8, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md8);
    case 9:        /* the 8-rows x 2-columns-per-lane consumers (A/B against k_sweep_quad) */
      if (C == 32) return launch_sweep_shape<64, 64, 2, 8, 32>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);
      if (C == 16) return launch_sweep_shape<64, 64, 3, 8, 16>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);
      return launch_sweep_shape<64, 64, 4, 8, 8>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);
    default:
      if (C == 32) return launch_sweep_quad<2, 32>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);
      if (C == 16) return launch_sweep_quad<3, 16>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);
      return launch_sweep_quad<4, 8>(g, b, m, mK, mKS, dst, slot0, view, counters, np_ub, grid, s, md);
  }
}
cudaError_t ekf_launch_end_scan(const EkfGeom& g, const EkfBuffers& b, const double* d_z, const double* d_R,
                                int m, int L_ub, int slot0, EkfScanView* view, cudaStream_t s,
                                double* P2, int prev_slot0, const int* prev_cnt_ptr) {
  /* all blocks of phase A redo the (idempotent) no-match bookkeeping only in thread 0 of block 0's
   * shared copy; to keep it race-free phase A runs as ONE block when it also has to write the pose */
  k_end_scan_a<<<1, 512, 0, s>>>(g, b, d_z, d_R, m, slot0, view, prev_slot0, prev_cnt_ptr);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if (m > 0) {
    const int cols_ub = 2 * ((m < g.cap) ? m : g.cap);
    int rows_ub = 3 + 2 * L_ub + 2 * m;
    if (rows_ub > g.n) rows_ub = g.n;
    int gy = rows_ub / 8; if (gy < 1) gy = 1; if (gy > 2048) gy = 2048;
    dim3 grid((cols_ub + EKF_BLOCK - 1) / EKF_BLOCK, gy);
    k_end_scan_b<<<grid, EKF_BLOCK, 0, s>>>(g, b, P2);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}
cudaError_t ekf_launch_assemble(const EkfGeom& g, const EkfBuffers& b, int r0, int nr, int c0, int nc,
                                double* d_out, int ld_out, cudaStream_t s) {
  k_assemble<<<blocks_for((long long)nr * nc, 148 * 16), EKF_BLOCK, 0, s>>>(g, b, r0, nr, c0, nc, d_out, ld_out);
  return cudaGetLastError();
}
cudaError_t ekf_launch_scatter(const EkfGeom& g, const EkfBuffers& b, int r0, int nr, int nl, const double* d_in,
                               int ld_in, cudaStream_t s) {
  k_scatter<<<blocks_for((long long)nr * nl, 148 * 16), EKF_BLOCK, 0, s>>>(g, b, r0, nr, nl, d_in, ld_in);
  return cudaGetLastError();
}
cudaError_t ekf_launch_cov_stats(const EkfGeom& g, const EkfBuffers& b, double* d_partials, int n_partials,
                                 double* d_out3, cudaStream_t s) {
  int grid = n_partials < 148 * 8 ? n_partials : 148 * 8;
  if (grid < 1) grid = 1;
  k_cov_rows<<<grid, EKF_BLOCK, 0, s>>>(g, b, d_partials);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  k_cov_fold<<<1, 32, 0, s>>>(b, d_partials, d_out3);
  return cudaGetLastError();
}
cudaError_t ekf_launch_remove_hot(const EkfGeom& g, const EkfBuffers& b, const int* keep, int nl, double* stage, int put,
                                  cudaStream_t s) {
  k_remove_hot<<<blocks_for(6LL * nl, 148 * 8), EKF_BLOCK, 0, s>>>(g, b, keep, nl, stage, put);
  return cudaGetLastError();
}
cudaError_t ekf_launch_remove_cold(const double* src, size_t ld_src, int src_row0, double* dst, size_t ld_dst, int dst_row0,
                                   const int* keep, int r0, int nr, int nl, int c_from, cudaStream_t s) {
  if (nr <= 0) return cudaSuccess;
  if (keep) k_remove_cold<true><<<nr, EKF_BLOCK, 0, s>>>(src, ld_src, src_row0, dst, ld_dst, dst_row0, keep, r0, nr, nl, c_from);
  else k_remove_cold<false><<<nr, EKF_BLOCK, 0, s>>>(src, ld_src, src_row0, dst, ld_dst, dst_row0, keep, r0, nr, nl, c_from);
  return cudaGetLastError();
}
cudaError_t ekf_launch_insert_hot(const EkfGeom& g, const EkfBuffers& b, int L, int k, const double* src, cudaStream_t s) {
  if (k <= 0) return cudaSuccess;
  k_insert_hot<<<blocks_for(k, 148 * 8), EKF_BLOCK, 0, s>>>(g, b, L, k, src);
  return cudaGetLastError();
}
cudaError_t ekf_launch_insert_cold(double* P, size_t ld, int nl_old, int nl, int r0, int nr, const double* blk, int blk_row0,
                                   cudaStream_t s) {
  if (nr <= 0 || nl <= nl_old) return cudaSuccess;
  k_insert_cold<<<nr, EKF_BLOCK, 0, s>>>(P, ld, nl_old, nl, r0, nr, blk, blk_row0);
  return cudaGetLastError();
}
cudaError_t ekf_launch_pose_gain(const EkfGeom& g, const EkfBuffers& b, const EkfPoseFix& f, int d, double2* K2,
                                 double2* KS2, int L_ub, cudaStream_t s) {
  const int grid = blocks_for(3 + 2LL * L_ub, 148 * 8);
  if (d == 1) k_pose_gain<1><<<grid, EKF_BLOCK, 0, s>>>(g, b, f, K2, KS2);
  else if (d == 2) k_pose_gain<2><<<grid, EKF_BLOCK, 0, s>>>(g, b, f, K2, KS2);
  else if (d == 3) k_pose_gain<3><<<grid, EKF_BLOCK, 0, s>>>(g, b, f, K2, KS2);
  else return cudaErrorInvalidValue;
  return cudaGetLastError();
}
cudaError_t ekf_launch_pose_apply(const EkfGeom& g, const EkfBuffers& b, int d, const double2* K2, const double2* KS2,
                                  int max_np, int L_ub, cudaStream_t s) {
  const int grid = blocks_for(2LL * L_ub + 1, 148 * 8);
  if (d == 1) k_pose_apply<1><<<grid, EKF_BLOCK, 0, s>>>(g, b, K2, KS2, max_np);
  else if (d == 2) k_pose_apply<2><<<grid, EKF_BLOCK, 0, s>>>(g, b, K2, KS2, max_np);
  else if (d == 3) k_pose_apply<3><<<grid, EKF_BLOCK, 0, s>>>(g, b, K2, KS2, max_np);
  else return cudaErrorInvalidValue;
  return cudaGetLastError();
}
cudaError_t ekf_launch_pose_term2(const EkfGeom& g, const EkfBuffers& b, int d, const double2* K2, const double2* KS2,
                                  int L_ub, cudaStream_t s) {
  k_pose_term2<<<blocks_for(3 + 2LL * L_ub, 148 * 8), EKF_BLOCK, 0, s>>>(g, b, d, K2, KS2);
  return cudaGetLastError();
}
cudaError_t ekf_launch_zero_pending(const EkfGeom& g, const EkfBuffers& b, int m, int* d_np, cudaStream_t s) {
  k_zero_pending<<<blocks_for((long long)m * g.ld, 148 * 8), EKF_BLOCK, 0, s>>>(g, b, m, d_np);
  return cudaGetLastError();
}
