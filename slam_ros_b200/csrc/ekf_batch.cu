/* ekf_batch.cu -- independent filter instances (Monte-Carlo batches, BASELINE.json configs[3]).
 *
 * One thread block per filter; the whole Robot::localize (slam_ros/Robot.cpp:126-943) of that filter runs inside
 * one kernel launch with the filter's ENTIRE covariance in shared memory:
 *
 *   - storage, in HBM and in shared memory alike, is the upper triangle packed by COLUMNS: P[r,q] (r <= q) lives at
 *     q (q+1) / 2 + r.  The live part (columns < 3 + 2 L) is then a contiguous prefix whatever the capacity, and
 *     appending a landmark appends two columns at its end: a scan is ONE bulk copy in (cp.async.bulk, 43 KB at 50
 *     landmarks), the arithmetic, ONE bulk copy out -- 8 nl (nl+1) bytes of HBM traffic per filter and scan, and no
 *     global-memory round trip anywhere inside the scan;
 *   - with P on chip nothing has to be deferred: each matched line updates every element at once,
 *     p <- p - (K S)[r] K[q] (Robot.cpp:564-568), which is the reference's own order of operations;
 *   - association (Robot.cpp:313-501): every landmark first takes a test that needs no trigonometry and no matrix
 *     inverse -- the angle innovation alone bounds the Mahalanobis distance from below, d^2 >= v0^2 / S00 -- and is
 *     rejected when even that bound is twice the gate; the few survivors (typically one) are compacted onto the first
 *     lanes of one warp and evaluated by the reference's full expression; first fit = lowest passing index.  That warp
 *     works on the NEXT line's association while the other warps apply the previous match to the bulk of P.
 *
 * Filters never communicate; a multi-GPU batch is N independent ekf_batch objects, one per device
 * (slam_ros_b200/parallel.py deals filters round-robin).
 */
#include "../../include/ekf.h"
#include "ekf_internal.h"
#include "ekf_device.cuh"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define EKFB_THREADS 128
#ifndef EKFB_MIN_CTAS
#define EKFB_MIN_CTAS 4           /* CTAs per SM the register budget is cut for (4 x 128 threads x 128 registers = the whole file) */
#endif

struct EkfBatchState {
  double pose[3];
  int L;
  int sticky;
  int resets;
  int pad;
};

struct EkfBatchGeom {
  double2* scratch;         /* [B][4][n]: the pending gains of filters that run off chip */
  unsigned* sm_turn;        /* [256]: per SM, CTAs started there so far -- deals the association warp round-robin over the schedulers */
  EkfBatchState* st_out;    /* [B] or NULL: this launch's copy of the filters' records (the pipelined host path reads it back while the
                               next step's kernel already runs on the records themselves) */
  int B, cap, n, headroom;
  double gate, enc_noise, gate_d2max;
  long long pstride;        /* doubles per filter in the packed covariance array (even: 16-byte aligned filters) */
  int ystride;              /* doubles per filter in the state array (even) */
  int full_gates;           /* A/B: evaluate the full gate for every landmark (no lower-bound pre-test) */
};

namespace {

__host__ __device__ inline int tri(int q) { return (q * (q + 1)) >> 1; }        /* first element of packed column q */

/* shared-memory carve-up: the packed triangle holds columns < ns (a HINT: the largest map the host last saw, plus a
 * little; a filter that has outgrown it works on its HBM copy instead -- slower, same bits); y and the gain vectors
 * are sized by the capacity */
struct BatchLayout { int P, y, K, KS, zr, ext, matched, bytes; };
__host__ __device__ inline BatchLayout batch_layout(int ns, int n, int cap, int m) {
  BatchLayout l;
  int o = 0;
  l.P = o; o += ((tri(ns) + 1) & ~1) * 8;            /* packed upper triangle, columns < ns */
  l.y = o; o += ((n + 1) & ~1) * 8;
  l.K = o; o += 2 * ns * 16;                         /* two pending gains: K, then K S (off-chip filters: HBM scratch) */
  l.KS = o; o += 2 * ns * 16;
  l.zr = o; o += 6 * m * 8;                          /* the scan's lines: z (2 m), then R (4 m) */
  l.ext = o; o += ((m + 3) & ~3) * 4;
  l.matched = o; o += (cap + 15) & ~15;
  l.bytes = o;
  return l;
}

__device__ __forceinline__ unsigned b_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void b_mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(b_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void b_mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void b_mbar_wait(unsigned long long* bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "B_WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra B_WAIT_DONE;\n"
      "bra B_WAIT_LOOP;\n"
      "B_WAIT_DONE:\n"
      "}\n" ::"r"(b_smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void b_bulk_load(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(b_smem_u32(dst)), "l"(src), "r"(bytes), "r"(b_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void b_bulk_store(void* dst, const void* src, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(b_smem_u32(src)), "r"(bytes) : "memory");
}

/* Robot.cpp:564-568 on the COLD elements of the packed upper triangle, p <- (p - (K S)_0[r] K_0[q]) - (K S)_1[r] K_1[q] for
 * one or two pending matches in their order: column q >= 3, rows 3 up to (excluding) its landmark's 2x2 diagonal block;
 * rows 0..2 and the diagonal blocks are the hot part (phase A of the line loop).
 *
 * Work is cut into bands of 32 rows: lane l of every warp owns row rb + l of the band and keeps that row's (K S) entries in
 * registers; the columns that reach the band are dealt round-robin to the warps, and a warp takes four of its columns per
 * step -- the four column gains and the four elements are loaded first, then updated, then stored, so that the shared-memory
 * latency and the dependent multiply-add pairs of four independent elements overlap.  Consecutive lanes touch consecutive
 * words of a packed column: conflict-free.  (The first form of this pass walked long/short column pairs with four rows per
 * lane; its per-pair address and predicate arithmetic made it 2.5 k instructions per warp and pass, issued at one per ~6
 * cycles -- the phase timers showed it, not the association gate beside it, bounding the line loop.)  Warp w0 of nw. */
template <bool TWO, int NW>
__device__ __forceinline__ void batch_update_cold_t(double* __restrict__ P, const double2* __restrict__ K0, const double2* __restrict__ KS0,
                                                    const double2* __restrict__ K1, const double2* __restrict__ KS1,
                                                    int nl, int qlo, int qhi, int w0, int lane) {
  /* columns [qlo, qhi) only (the line loop folds the triangle one half at a time): below, `qhi` bounds the columns */
  for (int rb = 0; rb + 2 < qhi; rb += 32) {         /* the last column's cold rows end at qhi - 3 */
    const int r = rb + lane;
    double2 a0 = make_double2(0.0, 0.0), a1 = a0;
    if (r < nl) { a0 = KS0[r]; if (TWO) a1 = KS1[r]; }
    const bool rok = r >= 3;
    /* Column q is cold above its landmark's diagonal block, rows < e(q) = (q - 1) | 1.  It reaches this band from
     * q = rb + 1 on and covers the whole band from q = rb + 33 on: only the columns in between need a per-row test. */
    int q = (rb + 1 > 3 ? rb + 1 : 3);
    if (q < qlo) q = qlo;
    q += w0;
    const int qfull = rb + 33 < qhi ? rb + 33 : qhi;
    /* tri(q + d) - tri(q) = d q + tri(d): the four columns of a step sit at e, e + (NW q + tri(NW)), ...  Everything is
     * taken four columns at a time -- loads, then the multiply-add pairs, then stores -- so that a step costs one
     * shared-memory latency and one dependent chain, not four; the ragged steps carry a per-column predicate. */
    double* e = P + tri(q) + r;
    const double2* k0p = K0 + q;
    const double2* k1p = K1 + q;
    const double2 zz = make_double2(0.0, 0.0);
#define EKFB_COLD_STEP(OK0, OK1, OK2, OK3)                                                                             \
    {                                                                                                                  \
      const int s1 = NW * q + tri(NW), s2 = 2 * NW * q + tri(2 * NW), s3 = 3 * NW * q + tri(3 * NW);                   \
      const bool o0 = (OK0), o1 = (OK1), o2 = (OK2), o3 = (OK3);                                                       \
      const double p0 = o0 ? e[0] : 0.0, p1 = o1 ? e[s1] : 0.0, p2 = o2 ? e[s2] : 0.0, p3 = o3 ? e[s3] : 0.0;          \
      const double2 g0 = o0 ? k0p[0] : zz, g1 = o1 ? k0p[NW] : zz, g2 = o2 ? k0p[2 * NW] : zz, g3 = o3 ? k0p[3 * NW] : zz; \
      double x0 = sub_rank2(p0, a0, g0), x1 = sub_rank2(p1, a0, g1), x2 = sub_rank2(p2, a0, g2), x3 = sub_rank2(p3, a0, g3); \
      if (TWO) {                                                                                                       \
        const double2 h0 = o0 ? k1p[0] : zz, h1 = o1 ? k1p[NW] : zz, h2 = o2 ? k1p[2 * NW] : zz, h3 = o3 ? k1p[3 * NW] : zz; \
        x0 = sub_rank2(x0, a1, h0); x1 = sub_rank2(x1, a1, h1); x2 = sub_rank2(x2, a1, h2); x3 = sub_rank2(x3, a1, h3); \
      }                                                                                                                \
      if (o0) e[0] = x0;                                                                                               \
      if (o1) e[s1] = x1;                                                                                              \
      if (o2) e[s2] = x2;                                                                                              \
      if (o3) e[s3] = x3;                                                                                              \
      e += 4 * NW * q + tri(4 * NW);                                                                                   \
      k0p += 4 * NW; k1p += 4 * NW;                                                                                    \
      q += 4 * NW;                                                                                                     \
    }
#define EKFB_COLD_OK(d) (rok && q + (d) < qhi && r < ((q + (d) - 1) | 1))
    while (q < qfull) EKFB_COLD_STEP(EKFB_COLD_OK(0), EKFB_COLD_OK(NW), EKFB_COLD_OK(2 * NW), EKFB_COLD_OK(3 * NW))
    if (rok) {
      while (q + 3 * NW < qhi) EKFB_COLD_STEP(true, true, true, true)
      if (q < qhi) EKFB_COLD_STEP(true, q + NW < qhi, q + 2 * NW < qhi, q + 3 * NW < qhi)
    }
#undef EKFB_COLD_OK
#undef EKFB_COLD_STEP
  }
}
/* nw is 3 beside an association (the fourth warp gates) and 4 after the scan's last line */
__device__ __forceinline__ void batch_update_cold(double* __restrict__ P, const double2* __restrict__ K0, const double2* __restrict__ KS0,
                                                  const double2* __restrict__ K1, const double2* __restrict__ KS1, bool two,
                                                  int nl, int qlo, int qhi, int w0, int nw, int lane) {
  if (nw == 3) {
    if (two) batch_update_cold_t<true, 3>(P, K0, KS0, K1, KS1, nl, qlo, qhi, w0, lane);
    else batch_update_cold_t<false, 3>(P, K0, KS0, K1, KS1, nl, qlo, qhi, w0, lane);
  } else {
    if (two) batch_update_cold_t<true, 4>(P, K0, KS0, K1, KS1, nl, qlo, qhi, w0, lane);
    else batch_update_cold_t<false, 4>(P, K0, KS0, K1, KS1, nl, qlo, qhi, w0, lane);
  }
}

/* The whole scan of one filter.  ns: columns of the packed triangle that fit the shared-memory carve-up. */
#ifdef EKFB_TIMING
#define BT_DECL long long bt_[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}; long long bt0_ = clock64()
#define BT_MARK(k) do { const long long n_ = clock64(); bt_[k] += n_ - bt0_; bt0_ = n_; } while (0)
#define BT_RESET() bt0_ = clock64()
#define BT_PRINT() do { if (blockIdx.x == 7 && (threadIdx.x == 0 || threadIdx.x == 32)) printf("k_batch_scan block 7 thread %d, cycles: load %lld predict %lld | per scan: A %lld, B(gate or cold pass) %lld, B-barrier %lld, C %lld (setup %lld, loads+correction %lld, gain %lld, stores %lld), C-barrier %lld | tail %lld | gate: pre-test %lld gather %lld gate_from_block %lld first-fit+publish %lld\n", (int)threadIdx.x, bt_[0], bt_[1], bt_[2], bt_[3] + bt_[12] + bt_[13] + bt_[14] + bt_[15], bt_[4], bt_[5] + bt_[8] + bt_[9] + bt_[10] + bt_[11], bt_[8], bt_[9], bt_[10], bt_[11], bt_[6], bt_[7], bt_[12], bt_[13], bt_[14], bt_[15]); } while (0)
#else
#define BT_DECL do { } while (0)
#define BT_MARK(k) do { } while (0)
#define BT_RESET() do { } while (0)
#define BT_PRINT() do { } while (0)
#endif

template <bool ON_CHIP>
__device__ __forceinline__ void batch_scan_body(const EkfBatchGeom& g, const int ns, double* __restrict__ Yg,
                                                double* __restrict__ Pg, EkfBatchState* __restrict__ Sg,
                                                const double* __restrict__ U, const double* __restrict__ Z,
                                                const double* __restrict__ Rm, const int m, int* __restrict__ Jout, const int L0) {
  extern __shared__ __align__(16) unsigned char braw[];
  const BatchLayout lay = batch_layout(ns, g.n, g.cap, m);
  double* const Psm = reinterpret_cast<double*>(braw + lay.P);
  double* const ys = reinterpret_cast<double*>(braw + lay.y);
  /* pending gains: slot k & 1 holds K and K S of the scan's k-th match */
  const int kn = ON_CHIP ? ns : g.n;
  double2* const Ks = ON_CHIP ? reinterpret_cast<double2*>(braw + lay.K) : g.scratch + (size_t)blockIdx.x * 4 * g.n;
  double2* const KSs = ON_CHIP ? reinterpret_cast<double2*>(braw + lay.KS) : Ks + 2 * (size_t)g.n;
  double* const zs = reinterpret_cast<double*>(braw + lay.zr);
  double* const Rs = zs + 2 * m;
  int* const ext = reinterpret_cast<int*>(braw + lay.ext);
  unsigned char* const matched = braw + lay.matched;
  __shared__ unsigned long long s_bar;
  __shared__ int s_best, s_sticky, s_gw;
  __shared__ int s_cand[32];                                 /* survivors of the pre-test, in index order */
  __shared__ double s_xpre[3];
  __shared__ double s_M[6];                                   /* Fu Q Fu' (upper triangle, packed by columns) */
  __shared__ Gate sG;

  const int tid = threadIdx.x, nt = EKFB_THREADS, lane = tid & 31, warp = tid >> 5;
  const int f = blockIdx.x;
  double* const Pf = Pg + (size_t)f * g.pstride;
  double* const yf = Yg + (size_t)f * g.ystride;
  EkfBatchState* const st = Sg + f;
  const double* const u = U + 3 * (size_t)f;
  const double* const z = Z + 2 * (size_t)m * f;
  const double* const R = Rm + 4 * (size_t)m * f;
  int* const jout = Jout ? Jout + (size_t)m * f : 0;

  BT_DECL;
  int L = L0;
  const int nl = 3 + 2 * L;
  const double pose0 = st->pose[0], pose1 = st->pose[1], pose2 = st->pose[2];
  /* the whole live triangle on chip -- or, for a filter that has outgrown the carve-up, its HBM copy in place */
  constexpr bool on_chip = ON_CHIP;
  double* const Ps = ON_CHIP ? Psm : Pf;
  /* ---- the filter's live covariance and state: two bulk copies, one barrier ---- */
  if (tid == 0) {
    const unsigned pbytes = on_chip ? (unsigned)(((tri(nl) + 1) & ~1) * 8) : 0u, ybytes = (unsigned)(((nl + 1) & ~1) * 8);
    b_mbar_init(&s_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    b_mbar_expect_tx(&s_bar, pbytes + ybytes);
    if (on_chip) b_bulk_load(Psm, Pf, pbytes, &s_bar);
    b_bulk_load(ys, yf, ybytes, &s_bar);
    s_sticky = 0;
    /* Which warp associates.  Warp w of every CTA issues from scheduler w of the SM; were the gate always on warp 0, one
     * scheduler's fp64 pipe would carry the trigonometry and divisions of all four resident filters while the other three
     * idle between cold passes.  The CTAs that start on an SM take the four warps in turn. */
    unsigned smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    s_gw = (int)(atomicAdd(&g.sm_turn[smid & 255u], 1u) & 3u);
  }
  for (int j = tid; j < g.cap; j += nt) matched[j] = 0;
  /* the scan's lines travel to shared memory under the bulk copies: a gate then starts from a 29-cycle load instead of an
   * L2 / HBM round trip at the head of every line's dependent chain */
  for (int k = tid; k < 6 * m; k += nt) zs[k] = (k < 2 * m) ? z[k] : R[k - 2 * m];
  /* ---- prediction, Robot.cpp:130-258 (SURVEY appendix A.2): everything that does not need the covariance -- the
   * trigonometry, Fu Q Fu' (:180-218, :250-258), x_pre -- is computed while the bulk copies are in flight ---- */
  const double u0 = u[0], u2 = u[2];
  const double ang = add_rn(pose2, __ddiv_rn(u2, 2.0));
  double ca, sa;
  cos_sin(ang, ca, sa);
  const double F02 = mul_rn(-u0, sa), F12 = mul_rn(u0, ca);
  if (tid == 0) {
    const double Fu[3][3] = {{ca, 0.0, __ddiv_rn(mul_rn(-u0, sa), 2.0)},
                             {sa, 1.0, __ddiv_rn(mul_rn(u0, ca), 2.0)},
                             {0.0, 0.0, 1.0}};
    const double qf = add_rn(__ddiv_rn(-1.0, add_rn(1.0, fabs(u0))), 1.0);
    const double Q[3] = {mul_rn(g.enc_noise, qf), mul_rn(mul_rn(2.0, g.enc_noise), qf), mul_rn(g.enc_noise, qf)};
    double FQ[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
    for (int k = 0; k < 3; ++k)
      for (int i = 0; i < 3; ++i) {
        const double t = mul_rn(1.0, Fu[i][k]);
        if (t != 0.0)
          for (int j = 0; j < 3; ++j) FQ[i][j] = add_rn(FQ[i][j], mul_rn(t, (j == k) ? Q[k] : 0.0));
      }
    for (int i = 0; i < 3; ++i)
      for (int j = i; j < 3; ++j) {
        double t = 0.0;
        for (int k = 0; k < 3; ++k) t = add_rn(t, mul_rn(FQ[i][k], Fu[j][k]));
        s_M[tri(j) + i] = add_rn(0.0, mul_rn(1.0, t));                /* added to the predicted 3x3 block below */
      }
    s_xpre[0] = add_rn(pose0, mul_rn(u0, ca));
    s_xpre[1] = add_rn(pose1, mul_rn(u0, sa));
    s_xpre[2] = add_rn(pose2, u2);
  }
  __syncthreads();
  b_mbar_wait(&s_bar, 0);
  BT_MARK(0);

  const int gw = s_gw;
  for (int q = 3 + tid; q < nl; q += nt) {                            /* :242 rows 0,1 */
    double* c = Ps + tri(q);
    const double p2 = c[2];
    double a0 = add_rn(0.0, c[0]); axpy_skip(a0, F02, p2);
    double a1 = add_rn(0.0, c[1]); axpy_skip(a1, F12, p2);
    c[0] = a0; c[1] = a1;
  }
  if (tid == 0) {
    double A[3][3], T[3][3], Pn[3][3];
    for (int i = 0; i < 3; ++i) for (int k = i; k < 3; ++k) { A[i][k] = Ps[tri(k) + i]; A[k][i] = A[i][k]; }
    for (int j = 0; j < 3; ++j) {
      double r0 = 0.0, r1 = 0.0, r2 = 0.0;
      axpy_skip(r0, 1.0, A[0][j]); axpy_skip(r1, 1.0, A[1][j]);
      axpy_skip(r0, F02, A[2][j]); axpy_skip(r1, F12, A[2][j]); axpy_skip(r2, 1.0, A[2][j]);
      T[0][j] = r0; T[1][j] = r1; T[2][j] = r2;
    }
    for (int i = 0; i < 3; ++i) {
      double c0 = 0.0; c0 = add_rn(c0, mul_rn(T[i][0], 1.0)); c0 = add_rn(c0, mul_rn(T[i][2], F02));
      double c1 = 0.0; c1 = add_rn(c1, mul_rn(T[i][1], 1.0)); c1 = add_rn(c1, mul_rn(T[i][2], F12));
      Pn[i][0] = add_rn(0.0, c0); Pn[i][1] = add_rn(0.0, c1); Pn[i][2] = T[i][2];
    }
    for (int i = 0; i < 3; ++i)
      for (int j = i; j < 3; ++j) Ps[tri(j) + i] = add_rn(Pn[i][j], s_M[tri(j) + i]);
  }
  __syncthreads();

  /* ---- the observed lines in order, Robot.cpp:298-645 ----
   * Per line, three phases separated by block barriers:
   *   A  (all warps)  the HOT part of the newest match's update: rows 0..2 of every column, the 2x2 diagonal blocks,
   *                   y, the pose -- everything a gate reads;
   *   B  warp 0       associates this line (pre-test of every landmark, full gate of the survivors, first fit), WHILE
   *      warps 1..3   fold the pending matches into the cold rest of the triangle -- two at a time: a match's cold update
   *                   waits for the next match, so that P is read and written once per TWO rank-2 terms;
   *   C  (all warps)  the gain rows of this line's match; a column entry whose pending term is not folded yet is
   *                   corrected on the fly (same operations, same order).
   * The long dependent chain of a gate (trigonometry, 2x2 LU inverse) thus runs beside the bulk of the update. */
  BT_MARK(1);
  int ne = 0, nmatch = 0;                                    /* uniform across the block */
  const double gate2x4 = 4.0 * g.gate * g.gate;
  /* The cold triangle is folded one HALF at a time: H0 = columns < qs, H1 = columns >= qs, qs ~ nl / sqrt 2 (equal work), odd
   * so that a landmark's two columns stay together.  np0 / np1: the most recent matches whose cold update is pending in H0 /
   * H1.  Beside EVERY gate the three other warps fold the half with more pending terms (both its terms: each element is
   * still read and written once per two rank-2 terms), so the cold work is the same every line instead of a full pass
   * beside every second gate -- which took longer than the gate and made the gate warp wait.  After a fold the other half
   * holds at most one pending term, so a gain row still corrects a column entry against at most one term, and a term is
   * folded everywhere before its slot is reused two matches later.  -DEKFB_FULL_PASS: the whole triangle beside every second
   * gate (A/B). */
#ifdef EKFB_FULL_PASS
  const int qs = nl;
#else
#ifndef EKFB_SPLIT
#define EKFB_SPLIT 0.7071f
#endif
  const int qs = min(nl, max(3, (int)(EKFB_SPLIT * (float)nl) | 1));
#endif
  int np0 = 0, np1 = 0, last_h = 1;
  bool have_new = false;                                     /* match nmatch-1: hot part pending too */
  for (int i = 0; i <= m; ++i) {
    const bool gating = i < m;
    if (!gating && np0 == 0 && np1 == 0) break;
    /* ---- phase A ---- */
    if (have_new) {
      const double2* Kn = Ks + (size_t)((nmatch - 1) & 1) * kn;
      const double2* KSn = KSs + (size_t)((nmatch - 1) & 1) * kn;
      const double v0 = sG.v[0], v1 = sG.v[1];
      const double2 ks0 = KSn[0], ks1 = KSn[1], ks2 = KSn[2];
      for (int q = tid; q < nl; q += nt) {
        double* c = Ps + tri(q);
        const double2 kq = Kn[q];
        if (q >= 3) {
          /* :564-568 on the column's hot entries -- rows 0..2 and the landmark's diagonal block -- all loaded first */
          const bool odd = q & 1;                                                    /* q = a: (a,a); q = b: (a,b), (b,b) */
          const double2 ksq = KSn[q], ksp = KSn[q - 1];
          const double c0 = c[0], c1 = c[1], c2 = c[2], cq = c[q], cp = c[q - 1];
          c[0] = sub_rank2(c0, ks0, kq); c[1] = sub_rank2(c1, ks1, kq); c[2] = sub_rank2(c2, ks2, kq);
          c[q] = sub_rank2(cq, ksq, kq);
          if (!odd) c[q - 1] = sub_rank2(cp, ksp, kq);
          double t = 0.0;                                                            /* :585-589  y += K * delta */
          axpy_skip(t, kq.x, v0); axpy_skip(t, kq.y, v1);
          ys[q] = add_rn(ys[q], t);
        } else {
          for (int r = 0; r <= q; ++r) c[r] = sub_rank2(c[r], KSn[r], kq);           /* the robot block's upper triangle */
        }
      }
      if (tid == nt - 1) {            /* the robot pose: on the last thread, which has no column of its own up to 127 rows */
        double yn[3];
        for (int r = 0; r < 3; ++r) {
          const double2 kk = Kn[r];
          double t = 0.0;
          axpy_skip(t, kk.x, v0); axpy_skip(t, kk.y, v1);
          yn[r] = add_rn(s_xpre[r], t);
        }
        normalize_radian(yn[2]);                                      /* :596-602 */
        for (int r = 0; r < 3; ++r) { ys[r] = yn[r]; s_xpre[r] = yn[r]; }
      }
      have_new = false;
      __syncthreads();
    }
    BT_MARK(2);
    /* ---- phase B ---- */
    int fh = -1;                                               /* the half folded beside this line's gate */
    if (gating) {
#ifdef EKFB_FULL_PASS
      if (np0 == 2) fh = 0;
#else
      if (np0 > np1 || (np0 == np1 && np0 > 0 && last_h == 1)) fh = 0;
      else if (np1 > 0) fh = 1;
#endif
    }
    /* fold of half h: its np_h most recent matches, the older first */
    auto cold_half = [&](int h, int w0, int nw) {
      const int n = h ? np1 : np0;
      const int s0 = (nmatch - n) & 1;
      batch_update_cold(Ps, Ks + (size_t)s0 * kn, KSs + (size_t)s0 * kn, Ks + (size_t)(s0 ^ 1) * kn, KSs + (size_t)(s0 ^ 1) * kn,
                        n == 2, nl, h ? qs : 3, h ? nl : qs, w0, nw, lane);
    };
    if (warp == gw && gating) {
      const double z0 = zs[2 * i], z1 = zs[2 * i + 1];
      const double Rl[4] = {Rs[4 * i], Rs[4 * i + 1], Rs[4 * i + 2], Rs[4 * i + 3]};
      const double xp[3] = {s_xpre[0], s_xpre[1], s_xpre[2]};
      const double P22 = Ps[tri(2) + 2];
      int best = EKF_NO_MATCH, sing = EKF_NO_MATCH;                   /* sing: this lane's lowest singular pair */
      int j0 = 0;
      while (j0 < L && best == EKF_NO_MATCH) {                        /* first fit: a match among these candidates ends the search */
        /* rounds of 32 landmarks take the pre-test; their survivors, in index order, fill the lanes of ONE round of full
         * gates (typically one or two survivors out of 50 landmarks: one trigonometry + LU chain per line, not one per
         * 32 landmarks) */
        int ncand = 0;
        while (j0 < L) {
          /* pre-test of two rounds of 32 landmarks at once, straight-line code (their loads and chains interleave).
           * v is the angle innovation of Robot.cpp:423-475 as its representative of least magnitude, w - 2 pi rint(w / 2 pi)
           * -- within rounding of, or smaller than, what the reference's wraps leave -- and S00 = H0 P H0' + R00 with
           * H0 = (0, 0, -1, .. 1 at a ..): d^2 = v' S^-1 v >= v^2 / S00, so a landmark whose bound exceeds (2 gate)^2 --
           * twice the gate in d, far outside any rounding difference between the bound and the reference's LU
           * expression -- cannot pass the reference's test either */
          bool keep[2];
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int j = j0 + 32 * h + lane;
            const bool live = j < L;
            const int a = live ? 3 + 2 * j : 3;
            const double* ca_ = Ps + tri(a);
            const bool free_ = live && !matched[live ? j : 0];
            const double w = sub_rn(z0, sub_rn(ys[a], xp[2]));
            const double v = __fma_rn(-(2.0 * EKF_PI), rint(w * (1.0 / (2.0 * EKF_PI))), w);
            const double S00 = (P22 - 2.0 * ca_[2]) + ca_[a] + Rl[0];
            keep[h] = free_ && (g.full_gates || !(S00 > 0.0) || !(v * v > gate2x4 * S00));
          }
          bool full = false;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            if (full || j0 >= L) break;
            const unsigned mask = __ballot_sync(0xffffffffu, keep[h]);
            const int nk = __popc(mask);
            if (ncand + nk > 32) { full = true; break; }              /* these survivors wait for the next round of full gates */
            if (keep[h]) s_cand[ncand + __popc(mask & ((1u << lane) - 1u))] = j0 + lane;
            ncand += nk;
            j0 += 32;
          }
          if (full) break;
        }
        __syncwarp();
        const int jj = lane < ncand ? s_cand[lane] : 0;
        BT_MARK(12);
        int mine = EKF_NO_MATCH;
        Gate Gj;
        if (lane < ncand) {                                           /* the survivors, compacted onto the first lanes */
          const int a = 3 + 2 * jj, bb = a + 1;
          const double* ca_ = Ps + tri(a);
          const double* cb_ = Ps + tri(bb);
          double Cm[5][5];
          for (int r = 0; r < 3; ++r) {
            for (int q = r; q < 3; ++q) { Cm[r][q] = Ps[tri(q) + r]; Cm[q][r] = Cm[r][q]; }
            Cm[r][3] = Cm[3][r] = ca_[r]; Cm[r][4] = Cm[4][r] = cb_[r];
          }
          Cm[3][3] = ca_[a]; Cm[3][4] = Cm[4][3] = cb_[a]; Cm[4][4] = cb_[bb];
          BT_MARK(13);
          gate_from_block(Cm, ys[a], ys[bb], xp, z0, z1, Rl, Gj);
          if (Gj.singular) sing = min(sing, jj);
          else if (!gate_rejects_d2(Gj.d2, g.gate_d2max)) mine = jj;                   /* :489 */
          BT_MARK(14);
        }
        best = __reduce_min_sync(0xffffffffu, mine);
        if (mine != EKF_NO_MATCH && mine == best) sG = Gj;            /* the winner publishes its gate record */
        BT_MARK(15);
      }
      /* EKF_ESINGULAR: a singular pair that first fit skipped before its winner (any, when the line matched nothing) */
      sing = __reduce_min_sync(0xffffffffu, sing);
      if (lane == 0) {
        if (sing < best) atomicOr(&s_sticky, EKF_STICKY_SINGULAR);
        s_best = best;
        if (best == EKF_NO_MATCH) { ext[ne] = i; if (jout) jout[i] = -1; }           /* :309 / :325 / :493 */
        else { matched[best] = 1; if (jout) jout[i] = best; }                       /* :501 */
      }
    } else if (gating && fh >= 0) {
      cold_half(fh, (warp - gw - 1) & 3, nt / 32 - 1);
    } else if (!gating) {                                             /* after the last line: whatever is still pending, all warps */
      if (np0 > 0) cold_half(0, warp, nt / 32);
      if (np1 > 0) cold_half(1, warp, nt / 32);
    }
    BT_MARK(3);
    __syncthreads();
    BT_MARK(4);
    if (fh == 0) { np0 = 0; last_h = 0; }
    else if (fh == 1) { np1 = 0; last_h = 1; }
    if (!gating) break;
    const int jb = s_best;
    if (jb == EKF_NO_MATCH) { ne += 1; continue; }
    /* ---- phase C: Robot.cpp:516-560 ---- */
    {
      const int a = 3 + 2 * jb, bb = a + 1;
      const int ta = tri(a), tb = tri(bb);
      const double2* Kp = Ks + (size_t)((nmatch - 1) & 1) * kn;       /* the one match that may still be pending in a half */
      const double2* KSp = KSs + (size_t)((nmatch - 1) & 1) * kn;
      double2* Kw = Ks + (size_t)(nmatch & 1) * kn;
      double2* KSw = KSs + (size_t)(nmatch & 1) * kn;
      double2 kpa = make_double2(0.0, 0.0), kpb = kpa, kspa = kpa, kspb = kpa;
      if (np0 + np1 > 0) { kpa = Kp[a]; kpb = Kp[bb]; kspa = KSp[a]; kspb = KSp[bb]; }
      const bool pend_ca = (a >= qs ? np1 : np0) == 1, pend_cb = (bb >= qs ? np1 : np0) == 1;   /* columns a, b (rows above) */
      BT_MARK(8);
      for (int r = tid; r < nl; r += nt) {
        const int tr_ = tri(r);
        const double p0 = (r <= 0) ? Ps[r] : Ps[tr_];                 /* P[r,0..2] through the upper storage */
        const double p1 = (r <= 1) ? Ps[tri(1) + r] : Ps[tr_ + 1];
        const double p2 = (r <= 2) ? Ps[tri(2) + r] : Ps[tr_ + 2];
        double pa = (r <= a) ? Ps[ta + r] : Ps[tr_ + a];
        double pb = (r <= bb) ? Ps[tb + r] : Ps[tr_ + bb];
        if (r > 2 && r != a && r != bb) {                             /* cold entries: the pending term of their half, on the fly */
          if (r < a) {
            if (pend_ca || pend_cb) {
              const double2 ksr = KSp[r];
              if (pend_ca) pa = sub_rank2(pa, ksr, kpa);
              if (pend_cb) pb = sub_rank2(pb, ksr, kpb);
            }
          } else if ((r >= qs ? np1 : np0) == 1) {                    /* (a, r), (b, r) live in column r */
            const double2 kr = Kp[r];
            pa = sub_rank2(pa, kspa, kr); pb = sub_rank2(pb, kspb, kr);
          }
        }
        BT_MARK(9);
        double2 Kr, KSr;
        gain_row(sG, p0, p1, p2, pa, pb, Kr, KSr);
        BT_MARK(10);
        Kw[r] = Kr; KSw[r] = KSr;
        BT_MARK(11);
      }
    }
    nmatch += 1; np0 += 1; if (qs < nl) np1 += 1; have_new = true;
    BT_MARK(5);
    __syncthreads();
    BT_MARK(6);
  }
  BT_RESET();

  /* ---- Robot.cpp:702-716 ---- */
  const double ps0 = s_xpre[0], ps1 = s_xpre[1];
  double ps2 = s_xpre[2];
  if (m == 0 || nmatch == 0) {
    if (tid == 0) { ys[0] = ps0; ys[1] = ps1; ys[2] = ps2; }
    normalize_radian(ps2);
  }
  __syncthreads();

  /* ---- augmentation in queue order, Robot.cpp:776-866: two new packed columns per line ---- */
  for (int e = 0; e < ne; ++e) {
    if (L >= g.cap) { if (tid == 0) s_sticky |= EKF_STICKY_CAPACITY; break; }      /* the reference overruns y[] here (Q4) */
    const int l = 3 + 2 * L;
    const int i = ext[e];
    double alfa = zs[2 * i], rr = zs[2 * i + 1];
    rr = add_rn(rr, add_rn(mul_rn(ps0, cos(alfa)), mul_rn(ps1, sin(alfa))));          /* :792 (Q8) */
    alfa = add_rn(alfa, ps2);                                                       /* :793 */
    double cw, sw;
    cos_sin(alfa, cw, sw);
    /* a new column lives on chip while it fits the carve-up, else straight in the filter's HBM copy (write-mostly:
     * only its rows 0..2 are read again, by the columns appended after it in this scan) */
    double* c0 = ((on_chip && l < ns) ? Psm : Pf) + tri(l);
    double* c1 = ((on_chip && l + 1 < ns) ? Psm : Pf) + tri(l + 1);
    for (int k = tid; k < l; k += nt) {                               /* :856-860: P[k, l], P[k, l+1] */
      const double* ck = ((on_chip && k < ns) ? Psm : Pf) + tri(k);
      const double a0 = (k <= 0) ? Ps[k] : ck[0];                     /* P[0,k], P[1,k], P[2,k] through the upper storage */
      const double a1 = (k <= 1) ? Ps[tri(1) + k] : ck[1];
      const double a2 = (k <= 2) ? Ps[tri(2) + k] : ck[2];
      double r0 = 0.0, r1 = 0.0;
      axpy_skip(r1, cw, a0);
      axpy_skip(r1, sw, a1);
      axpy_skip(r0, 1.0, a2);
      c0[k] = r0; c1[k] = r1;
    }
    if (tid == 0) {
      const double Rl[4] = {Rs[4 * i], Rs[4 * i + 1], Rs[4 * i + 2], Rs[4 * i + 3]};
      const double Gx[2][3] = {{0.0, 0.0, 1.0}, {cw, sw, 0.0}};
      const double Gl[2][2] = {{1.0, 0.0}, {sub_rn(mul_rn(ys[1], cw), mul_rn(ys[0], sw)), 1.0}};   /* :797-798 */
      double an = alfa;
      normalize_radian(an);                                                         /* :801 */
      ys[l] = an; ys[l + 1] = rr;
      double A[3][3];
      for (int ii = 0; ii < 3; ++ii) for (int kk = ii; kk < 3; ++kk) { A[ii][kk] = Ps[tri(kk) + ii]; A[kk][ii] = A[ii][kk]; }
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
      c0[l] = Pll[0][0]; c1[l] = Pll[0][1]; c1[l + 1] = Pll[1][1];
    }
    L += 1;
    __syncthreads();
  }

  /* ---- reset, Robot.cpp:893-904 (dead entries are never read; downloads zero them) ---- */
  int resets = 0;
  if (L > g.cap - g.headroom) { L = 0; resets = 1; }
  const int nl_new = 3 + 2 * L;
  for (int q = nl_new + tid; q < g.ystride; q += nt) ys[q] = 0.0;    /* Robot::y is zero beyond the live part */
  /* ---- state and covariance back to HBM: one bulk store each ---- */
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  __syncthreads();
  if (tid == 0) {
    if (on_chip) b_bulk_store(Pf, Psm, (unsigned)(((tri(min(nl_new, ns)) + 1) & ~1) * 8));
    b_bulk_store(yf, ys, (unsigned)(g.ystride * 8));
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    st->L = L; st->pose[0] = ps0; st->pose[1] = ps1; st->pose[2] = ps2;
    st->sticky = s_sticky;                        /* status reports this scan only */
    st->resets += resets;
    if (g.st_out) {
      EkfBatchState o;
      o.pose[0] = ps0; o.pose[1] = ps1; o.pose[2] = ps2; o.L = L; o.sticky = s_sticky; o.resets = st->resets; o.pad = 0;
      g.st_out[f] = o;
    }
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   /* the shared-memory source has been read: the CTA may go */
  }
  BT_MARK(7);
  BT_PRINT();
}

/* Robot::localize for filter blockIdx.x */
__global__ void __launch_bounds__(EKFB_THREADS, EKFB_MIN_CTAS) k_batch_scan(EkfBatchGeom g, int ns, double* __restrict__ Yg,
                                                                double* __restrict__ Pg, EkfBatchState* __restrict__ Sg,
                                                                const double* __restrict__ U, const double* __restrict__ Z,
                                                                const double* __restrict__ Rm, int m, int* __restrict__ Jout) {
  const int L0 = Sg[blockIdx.x].L;
  if (3 + 2 * L0 <= ns) batch_scan_body<true>(g, ns, Yg, Pg, Sg, U, Z, Rm, m, Jout, L0);
  else batch_scan_body<false>(g, ns, Yg, Pg, Sg, U, Z, Rm, m, Jout, L0);
}

__global__ void k_batch_init(EkfBatchGeom g, double* Pg) {
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f < g.B) {
    double* Pf = Pg + (size_t)f * g.pstride;
    Pf[tri(0)] = 0.05; Pf[tri(1) + 1] = 0.05; Pf[tri(2) + 2] = 0.0;               /* Robot.cpp:27-30 */
  }
}

}  // namespace

struct ekf_batch {
  ekf_config cfg;
  EkfBatchGeom g;
  cudaStream_t stream;              /* kernels and read-backs */
  cudaStream_t cstream;             /* input copies of the pipelined host path (overlap the previous step's kernel) */
  double* d_y; double* d_P; EkfBatchState* d_st;
  double2* d_scratch;               /* pending gains of filters running off chip: [B][4][n] */
  unsigned* d_sm_turn;              /* [256] */
  int max_m;
  /* two staging slots: ekf_batch_scan uses slot 0; ekf_batch_submit / ekf_batch_collect alternate */
  double* d_in[2]; double* h_in[2];       /* [u (3B) | z (2 m B) | R (4 m B)] */
  int* d_jout[2]; int* h_jout[2];
  EkfBatchState* h_sts[2];
  EkfBatchState* d_sts[2];          /* per-slot copy of the records as the slot's kernel left them */
  cudaStream_t dstream;             /* read-backs of the pipelined host path (run under the next step's kernel) */
  cudaEvent_t ev_in[2], ev_done[2], ev_kernel[2];
  int slot_m[2];
  int head, inflight;               /* oldest submitted slot, submitted-but-not-collected steps (0..2) */
  EkfBatchState* h_st;
  double* h_P;                      /* pinned staging of one filter's packed covariance (ekf_batch_download) */
  int L_hint;                       /* largest map of the batch when the states were last read back (sizes the on-chip triangle) */
  int L_exact;                      /* no device-resident scan was enqueued since then */
  int ns_forced;                    /* EKF_BATCH_NS: test knob, columns of the on-chip triangle (0 = from L_hint) */
  size_t smem_set;
  char err[256];
};

namespace {
#define CUB(call)                                                                             \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) {                                                                  \
      snprintf(b->err, sizeof b->err, "%s:%d %s: %s", "ekf_batch.cu", __LINE__, #call, cudaGetErrorString(e_)); \
      return EKF_ECUDA;                                                                       \
    }                                                                                         \
  } while (0)

const size_t kBatchSmemMax = 227 * 1024 - 256;      /* dynamic shared memory one CTA may ask for (static part: ~200 B) */

/* Columns of the on-chip triangle: the largest map last seen plus two lines of slack.  Not a bound -- a filter whose
 * live dimension exceeds it runs the same kernel on its HBM copy -- so device-resident scans enqueued back to back
 * keep the small carve-up (4 filters per SM at 50 landmarks) instead of drifting to the capacity. */
int batch_ns(const ekf_batch* b) {
  long long l = (long long)b->L_hint + 2;
  if (b->ns_forced > 0) l = (b->ns_forced - 3) / 2;
  /* an even number of lines: the packed prefix then has an even number of doubles, so the 16-byte granularity of the
   * bulk copies never reaches into the first column kept off chip */
  l += l & 1;
  if (l > b->g.cap + 1) l = (b->g.cap + 1) & ~1;
  return 3 + 2 * (int)l;
}

int batch_ensure_m(ekf_batch* b, int m) {
  if (m <= b->max_m) return EKF_OK;
  /* nothing is released before the larger scan is known to fit: a rejected call leaves the batch usable */
  int cap = b->max_m > 0 ? b->max_m : 8;
  while (cap < m) cap *= 2;
  if ((size_t)batch_layout(3, b->g.n, b->g.cap, cap).bytes > kBatchSmemMax) cap = m;    /* do not reject m over the rounding */
  if ((size_t)batch_layout(3, b->g.n, b->g.cap, cap).bytes > kBatchSmemMax) {
    snprintf(b->err, sizeof b->err, "scan of %d lines does not fit shared memory", m);
    return EKF_EINVAL;
  }
  if (b->inflight) { snprintf(b->err, sizeof b->err, "a scan with more lines than any before (%d) while steps are in flight: collect them first", m); return EKF_ESTATE; }
  CUB(cudaStreamSynchronize(b->stream));
  CUB(cudaStreamSynchronize(b->cstream));
  CUB(cudaStreamSynchronize(b->dstream));
  b->max_m = 0;                       /* until every buffer below exists, the next call must come back here */
  const size_t B = b->g.B;
  for (int k = 0; k < 2; ++k) {
    cudaFree(b->d_in[k]); cudaFree(b->d_jout[k]); cudaFreeHost(b->h_in[k]); cudaFreeHost(b->h_jout[k]);
    b->d_in[k] = 0; b->d_jout[k] = 0; b->h_in[k] = 0; b->h_jout[k] = 0;
  }
  for (int k = 0; k < 2; ++k) {
    CUB(cudaMalloc(&b->d_in[k], (3 + 6 * (size_t)cap) * B * sizeof(double)));
    CUB(cudaMallocHost(&b->h_in[k], (3 + 6 * (size_t)cap) * B * sizeof(double)));
    CUB(cudaMalloc(&b->d_jout[k], (size_t)cap * B * sizeof(int)));
    CUB(cudaMallocHost(&b->h_jout[k], (size_t)cap * B * sizeof(int)));
  }
  b->max_m = cap;
  return EKF_OK;
}

int batch_launch(ekf_batch* b, const double* d_u, int m, const double* d_z, const double* d_R, int* d_jout, EkfBatchState* d_st_out = 0) {
  int ns = batch_ns(b);
  while (ns > 3 && (size_t)batch_layout(ns, b->g.n, b->g.cap, m).bytes > kBatchSmemMax) ns -= 4;   /* very large maps: partly off chip */
  const size_t smem = (size_t)batch_layout(ns, b->g.n, b->g.cap, m).bytes;
  if (smem > kBatchSmemMax) { snprintf(b->err, sizeof b->err, "scan of %d lines does not fit shared memory", m); return EKF_EINVAL; }
  if (smem > b->smem_set) {
    CUB(cudaFuncSetAttribute(k_batch_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUB(cudaFuncSetAttribute(k_batch_scan, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    b->smem_set = smem;
  }
  EkfBatchGeom gl = b->g;
  gl.st_out = d_st_out;
  k_batch_scan<<<gl.B, EKFB_THREADS, smem, b->stream>>>(gl, ns, b->d_y, b->d_P, b->d_st, d_u, d_z, d_R, m, d_jout);
  CUB(cudaGetLastError());
  b->L_exact = 0;
  return EKF_OK;
}

/* after a synchronisation: the exact largest map of the batch (B small records) */
int batch_refresh_bound(ekf_batch* b) {
  if (b->L_exact) return EKF_OK;
  const size_t B = b->g.B;
  CUB(cudaMemcpyAsync(b->h_st, b->d_st, B * sizeof(EkfBatchState), cudaMemcpyDeviceToHost, b->stream));
  CUB(cudaStreamSynchronize(b->stream));
  int mx = 0;
  for (size_t f = 0; f < B; ++f) if (b->h_st[f].L > mx) mx = b->h_st[f].L;
  b->L_hint = mx; b->L_exact = 1;
  return EKF_OK;
}
}  // namespace

extern "C" {

int ekf_batch_create(ekf_batch** out, const ekf_config* cfg, int n_filters) {
  if (!out || !cfg || n_filters < 1 || cfg->capacity_lines < 1) return EKF_EINVAL;
  ekf_batch* b = new ekf_batch();
  memset(b, 0, sizeof *b);
  b->cfg = *cfg;
  *out = b;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    snprintf(b->err, sizeof b->err, "no CUDA device: libekfcuda has no CPU fallback");
    return EKF_ECUDA;
  }
  CUB(cudaSetDevice(cfg->device));
  EkfBatchGeom& g = b->g;
  g.B = n_filters; g.cap = cfg->capacity_lines; g.n = 3 + 2 * g.cap; g.headroom = cfg->reset_headroom;
  g.gate = cfg->gate; g.enc_noise = cfg->encoder_noise; g.gate_d2max = ekf_gate_d2max(cfg->gate);
  g.pstride = (tri(g.n) + 2) & ~1;
  g.ystride = (g.n + 1) & ~1;
  g.full_gates = (cfg->flags & EKF_FLAG_FULL_GATES) ? 1 : 0;
  if (g.cap > 2048 || (size_t)batch_layout(3, g.n, g.cap, 8).bytes > kBatchSmemMax) {
    snprintf(b->err, sizeof b->err, "capacity %d is too large for a batch filter (state and gain vectors are kept on chip); use ekf_create", g.cap);
    return EKF_EINVAL;
  }
  { const char* e = getenv("EKF_BATCH_NS"); b->ns_forced = e ? atoi(e) : 0; if (b->ns_forced < 0) b->ns_forced = 0; if (b->ns_forced > 0 && b->ns_forced < 3) b->ns_forced = 3; }
  CUB(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
  CUB(cudaStreamCreateWithFlags(&b->cstream, cudaStreamNonBlocking));
  CUB(cudaStreamCreateWithFlags(&b->dstream, cudaStreamNonBlocking));
  const size_t B = g.B;
  for (int k = 0; k < 2; ++k) {
    CUB(cudaEventCreateWithFlags(&b->ev_in[k], cudaEventDisableTiming));
    CUB(cudaEventCreateWithFlags(&b->ev_done[k], cudaEventDisableTiming));
    CUB(cudaEventCreateWithFlags(&b->ev_kernel[k], cudaEventDisableTiming));
    CUB(cudaMallocHost(&b->h_sts[k], B * sizeof(EkfBatchState)));
    CUB(cudaMalloc(&b->d_sts[k], B * sizeof(EkfBatchState)));
  }
  CUB(cudaMalloc(&b->d_y, B * (size_t)g.ystride * sizeof(double)));
  CUB(cudaMalloc(&b->d_P, B * (size_t)g.pstride * sizeof(double)));
  CUB(cudaMalloc(&b->d_st, B * sizeof(EkfBatchState)));
  CUB(cudaMalloc(&b->d_scratch, B * 4 * (size_t)g.n * sizeof(double2)));
  g.scratch = b->d_scratch;
  CUB(cudaMalloc(&b->d_sm_turn, 256 * sizeof(unsigned)));
  CUB(cudaMemsetAsync(b->d_sm_turn, 0, 256 * sizeof(unsigned), b->stream));
  g.sm_turn = b->d_sm_turn;
  CUB(cudaMallocHost(&b->h_st, B * sizeof(EkfBatchState)));
  CUB(cudaMallocHost(&b->h_P, (size_t)g.pstride * sizeof(double)));
  CUB(cudaMemsetAsync(b->d_y, 0, B * (size_t)g.ystride * sizeof(double), b->stream));
  CUB(cudaMemsetAsync(b->d_P, 0, B * (size_t)g.pstride * sizeof(double), b->stream));
  CUB(cudaMemsetAsync(b->d_st, 0, B * sizeof(EkfBatchState), b->stream));
  k_batch_init<<<(g.B + 255) / 256, 256, 0, b->stream>>>(g, b->d_P);
  CUB(cudaGetLastError());
  b->L_hint = 0; b->L_exact = 1;
  int rc = batch_ensure_m(b, 8);
  if (rc) return rc;
  CUB(cudaStreamSynchronize(b->stream));
  return EKF_OK;
}

int ekf_batch_destroy(ekf_batch* b) {
  if (!b) return EKF_EINVAL;
  cudaSetDevice(b->cfg.device);
  if (b->stream) cudaStreamSynchronize(b->stream);
  if (b->cstream) cudaStreamSynchronize(b->cstream);
  if (b->dstream) cudaStreamSynchronize(b->dstream);
  cudaFree(b->d_y); cudaFree(b->d_P); cudaFree(b->d_st); cudaFree(b->d_scratch); cudaFree(b->d_sm_turn);
  for (int k = 0; k < 2; ++k) {
    cudaFree(b->d_in[k]); cudaFree(b->d_jout[k]); cudaFreeHost(b->h_in[k]); cudaFreeHost(b->h_jout[k]); cudaFreeHost(b->h_sts[k]);
    if (b->ev_in[k]) cudaEventDestroy(b->ev_in[k]);
    if (b->ev_done[k]) cudaEventDestroy(b->ev_done[k]);
    if (b->ev_kernel[k]) cudaEventDestroy(b->ev_kernel[k]);
    cudaFree(b->d_sts[k]);
  }
  cudaFreeHost(b->h_st); cudaFreeHost(b->h_P);
  if (b->stream) cudaStreamDestroy(b->stream);
  if (b->cstream) cudaStreamDestroy(b->cstream);
  if (b->dstream) cudaStreamDestroy(b->dstream);
  delete b;
  return EKF_OK;
}

const char* ekf_batch_last_error(const ekf_batch* b) { return b ? b->err : "null batch"; }

int ekf_batch_scan_device(ekf_batch* b, const double* d_u, int m, const double* d_z, const double* d_R, int* d_j_out) {
  if (!b || !d_u || m < 0 || (m > 0 && (!d_z || !d_R))) return EKF_EINVAL;
  CUB(cudaSetDevice(b->cfg.device));
  return batch_launch(b, d_u, m, d_z, d_R, d_j_out);
}

/* Pipelined host path.  ekf_batch_submit copies one step's inputs into a pinned staging slot and enqueues its H2D copy
 * (on the copy stream), the kernel and the read-back of the matches and states; it returns at once.  Two steps may be
 * in flight: the inputs of step s+1 travel while the kernel of step s runs.  ekf_batch_collect waits for the OLDEST
 * submitted step. */
int ekf_batch_submit(ekf_batch* b, const double* u, int m, const double* z, const double* R) {
  if (!b || !u || m < 0 || (m > 0 && (!z || !R))) return EKF_EINVAL;
  if (b->inflight >= 2) { snprintf(b->err, sizeof b->err, "two steps are already in flight: ekf_batch_collect first"); return EKF_ESTATE; }
  CUB(cudaSetDevice(b->cfg.device));
  int rc = batch_ensure_m(b, m);
  if (rc) return rc;
  const int k = (b->head + b->inflight) & 1;
  const size_t B = b->g.B;
  double* h = b->h_in[k];
  memcpy(h, u, 3 * B * sizeof(double));
  if (m > 0) {
    memcpy(h + 3 * B, z, 2 * (size_t)m * B * sizeof(double));
    memcpy(h + 3 * B + 2 * (size_t)m * B, R, 4 * (size_t)m * B * sizeof(double));
  }
  const size_t total = (3 + 6 * (size_t)m) * B;
  CUB(cudaMemcpyAsync(b->d_in[k], h, total * sizeof(double), cudaMemcpyHostToDevice, b->cstream));
  CUB(cudaEventRecord(b->ev_in[k], b->cstream));
  CUB(cudaStreamWaitEvent(b->stream, b->ev_in[k], 0));
  rc = batch_launch(b, b->d_in[k], m, b->d_in[k] + 3 * B, b->d_in[k] + 3 * B + 2 * (size_t)m * B, b->d_jout[k], b->d_sts[k]);
  if (rc) return rc;
  /* the matches and the slot's copy of the records travel back on a stream of their own: the next step's kernel follows
   * this one directly instead of waiting for the read-back */
  CUB(cudaEventRecord(b->ev_kernel[k], b->stream));
  CUB(cudaStreamWaitEvent(b->dstream, b->ev_kernel[k], 0));
  if (m > 0) CUB(cudaMemcpyAsync(b->h_jout[k], b->d_jout[k], (size_t)m * B * sizeof(int), cudaMemcpyDeviceToHost, b->dstream));
  CUB(cudaMemcpyAsync(b->h_sts[k], b->d_sts[k], B * sizeof(EkfBatchState), cudaMemcpyDeviceToHost, b->dstream));
  CUB(cudaEventRecord(b->ev_done[k], b->dstream));
  b->slot_m[k] = m;
  b->inflight += 1;
  return EKF_OK;
}

int ekf_batch_collect(ekf_batch* b, int* j_out, double* pose) {
  if (!b) return EKF_EINVAL;
  if (b->inflight <= 0) { snprintf(b->err, sizeof b->err, "ekf_batch_collect: nothing was submitted"); return EKF_ESTATE; }
  CUB(cudaSetDevice(b->cfg.device));
  const int k = b->head;
  CUB(cudaEventSynchronize(b->ev_done[k]));
  const size_t B = b->g.B;
  const int m = b->slot_m[k];
  if (j_out && m > 0) memcpy(j_out, b->h_jout[k], (size_t)m * B * sizeof(int));
  int status = EKF_OK, mx = 0;
  const EkfBatchState* hs = b->h_sts[k];
  for (size_t f = 0; f < B; ++f) {
    if (pose) memcpy(pose + 3 * f, hs[f].pose, 3 * sizeof(double));
    if (hs[f].L > mx) mx = hs[f].L;
    if (hs[f].sticky & EKF_STICKY_CAPACITY) status = EKF_ECAPACITY;
    else if ((hs[f].sticky & EKF_STICKY_SINGULAR) && status == EKF_OK) status = EKF_ESINGULAR;
  }
  b->head ^= 1;
  b->inflight -= 1;
  b->L_hint = mx;                     /* the largest map as of that step: sizes the on-chip triangle of the next launches */
  b->L_exact = b->inflight == 0;
  return status;
}

int ekf_batch_scan(ekf_batch* b, const double* u, int m, const double* z, const double* R, int* j_out, double* pose) {
  if (!b) return EKF_EINVAL;
  if (b->inflight) { snprintf(b->err, sizeof b->err, "ekf_batch_scan while submitted steps are in flight: collect them first"); return EKF_ESTATE; }
  const int rc = ekf_batch_submit(b, u, m, z, R);
  if (rc) return rc;
  return ekf_batch_collect(b, j_out, pose);
}

int ekf_batch_sync(ekf_batch* b) {
  if (!b) return EKF_EINVAL;
  CUB(cudaSetDevice(b->cfg.device));
  CUB(cudaStreamSynchronize(b->stream));
  return batch_refresh_bound(b);
}

int ekf_batch_download(ekf_batch* b, int filter, double* y, double* P, int* n_lines, double pose[3]) {
  if (!b || filter < 0 || filter >= b->g.B) return EKF_EINVAL;
  CUB(cudaSetDevice(b->cfg.device));
  const size_t n = b->g.n;
  if (y) CUB(cudaMemcpyAsync(y, b->d_y + (size_t)filter * b->g.ystride, n * sizeof(double), cudaMemcpyDeviceToHost, b->stream));
  if (P) CUB(cudaMemcpyAsync(b->h_P, b->d_P + (size_t)filter * b->g.pstride, (size_t)tri((int)n) * sizeof(double), cudaMemcpyDeviceToHost, b->stream));
  CUB(cudaMemcpyAsync(b->h_st, b->d_st + filter, sizeof(EkfBatchState), cudaMemcpyDeviceToHost, b->stream));
  CUB(cudaStreamSynchronize(b->stream));
  b->L_exact = 0;                     /* h_st[0] now holds one filter's record, not the batch's */
  if (n_lines) *n_lines = b->h_st[0].L;
  if (pose) memcpy(pose, b->h_st[0].pose, 3 * sizeof(double));
  /* the device keeps the upper triangle of the live part, packed by columns: unpack, mirror, zero the rest
   * (Robot::P_t0 layout) */
  const size_t nl = 3 + 2 * (size_t)b->h_st[0].L;
  if (P)
    for (size_t r = 0; r < n; ++r)
      for (size_t q = 0; q < n; ++q) {
        if (r >= nl || q >= nl) P[r * n + q] = 0.0;
        else { const size_t lo = r < q ? r : q, hi = r < q ? q : r; P[r * n + q] = b->h_P[hi * (hi + 1) / 2 + lo]; }
      }
  if (y) for (size_t r = nl; r < n; ++r) y[r] = 0.0;
  return EKF_OK;
}

}  /* extern "C" */
