/* ekf_internal.h -- shared between the kernels (ekf_kernels.cu) and the C ABI (ekf_api.cu).
 *
 * HBM layout of one filter (DESIGN.md section 3).  n = 3 + 2*capacity, ld = n rounded up to 256 doubles
 * (2 KB) so every sweep tile (64, 128 or 256 columns wide) lies inside a row.
 *
 *   y     [ld]            state vector (Robot.h:26)
 *   top   [3][ld]         rows 0..2 of P (robot rows), upper part authoritative            -- "hot"
 *   diag  [cap][4]        per landmark j: P[a,a], P[a,b], P[b,b], pad  (a = 3+2j, b = a+1) -- "hot"
 *   P     [rows][ld]      every other ("cold") element, UPPER triangle authoritative, row-major,
 *                         64-row tile rows; in the row-sharded mode a rank stores only the tile rows
 *                         rb with rb % world == rank (local row = (rb / world) * 64 + r % 64)
 *   Kp,KSp[slots][ld]     double2: the scan's pending gains K_i and K_i*S_i (rank-2 terms not yet
 *                         folded into the cold part); slots = max(max_batch, 2 * group), the overlapped
 *                         path's ring of two halves of `group` slots (ekf_api.cu, create_common)
 *
 * Hot elements are kept current after every matched line (O(n) work); the cold part is brought up
 * to date by ONE sweep per scan -- or per group of scans on the overlapped path -- that applies the
 * pending terms in order, ((P - u_1) - u_2) ..., which is the reference's per-element arithmetic
 * (Robot.cpp:564-568) with m times less HBM traffic.
 */
#ifndef EKF_INTERNAL_H
#define EKF_INTERNAL_H

#include <cuda_runtime.h>
#include <limits.h>

#define EKF_TILE 64
#define EKF_LD_ALIGN 256                /* ld is a multiple of the widest sweep tile (256 columns) */
#define EKF_NO_MATCH INT_MAX
#define EKF_STICKY_CAPACITY 1
#define EKF_STICKY_SINGULAR 2
#define EKF_STICKY_XCHG 4               /* a peer never arrived at the cross-GPU exchange (row-sharded mode) */

struct EkfDevState {          /* one per filter, in global memory */
  double pose[3];             /* xPos, yPos, thetaPos (Robot.h:54-56) */
  double x_pre[3];            /* Robot.cpp:148, refreshed at :600-602 */
  double v[2];                /* innovation of the line being applied (delta, Robot.cpp:550) */
  double S[4];                /* its innovation covariance incl. R (diagnostic tap) */
  int L;                      /* savedLineCount (Robot.h:28) */
  int epoch;                  /* scan counter; matched[j] == epoch <=> j in matchSavedIndexes */
  int sticky;                 /* EKF_STICKY_* seen since last read */
  int n_added;                /* landmarks appended by the last end-of-scan */
  int resets;                 /* map resets so far (Robot.cpp:893-904) */
  int pbase;                  /* matches of this scan already folded into P by a mid-scan flush */
  int np;                     /* pending rank-2 terms = pidx[line] - pbase */
  int xseq;                   /* row-sharded mode: matched lines exchanged over NVLink so far (same on every rank) */
  int L0;                     /* savedLineCount before the last end-of-scan's append (read by its phase B) */
  /* the last absolute pose fix (ekf_observe_pose, d = its component count): decision and diagnostic tap */
  int fix_status;             /* EKF_FIX_* */
  double fix_S[9];            /* S = H P H' + R_sel, d x d with row stride 3 */
  double fix_v[3];            /* innovation z_sel - y_sel, theta wrapped */
  double fix_d2;              /* v' S^-1 v */
};
#define EKF_FIX_REJECTED 0
#define EKF_FIX_ACCEPTED 1
#define EKF_FIX_SINGULAR 2

/* one absolute pose fix, by value in the kernel parameters (compacted on the host, so that the kernels index it with
 * constants only): sel[0..d) = the selected state indices (0 x, 1 y, 2 theta) in increasing order, z = z_sel, R = R_sel
 * (d x d, row stride 3) */
struct EkfPoseFix { double z[3]; double R[9]; double d2max; int sel[3]; };

/* what a scan's (possibly later, possibly concurrent) sweep needs to know about that scan */
struct EkfScanView { int cnt; int L; int pad[2]; };

/* row-sharded mode: every rank's exchange buffer as mapped into THIS process (CUDA IPC); [rank] is the local one */
struct EkfPeers { double* xchg[8]; int world, rank; };

/* geometry handed to every kernel by value */
struct EkfGeom {
  int cap;        /* capacity in lines */
  int n;          /* 3 + 2*cap */
  int ld;         /* padded leading dimension (multiple of 64) */
  int rank, world;
  double gate, enc_noise;
  int headroom;
  double gate_d2max;   /* largest |d2| that passes: sqrt(|d2|) > gate  <=>  |d2| > gate_d2max (ekf_gate_d2max) */
};

struct EkfBuffers {
  EkfDevState* st;
  double* y;
  double* top;
  double* diag;
  double* P;
  int* matched;
  double2* Kp;
  double2* KSp;
  double* gates;      /* [cap][16]: gate record (c,s,g,S,Sinv,v,d2) of every landmark that passed the current line's gate */
  double* colA;       /* sharded mode: exchanged H-column slices */
  double* colB;
  /* per-scan line tables, sized max_lines (+1 for the prefix counters) */
  int* jbest;         /* first-fit winner per line (EKF_NO_MATCH = none) */
  int* jsing;         /* lowest landmark whose pair with the line has a singular S (EKF_NO_MATCH = none) */
  int* jout;          /* matched landmark or -1 per line */
  int* pidx;          /* pidx[i] = matches before line i; pidx[m] = matches in the scan */
  int* eidx;          /* eidx[i] = unmatched lines before line i */
  int* ext;           /* ext[e] = index of the e-th unmatched line */
  double* ext_cs;     /* per unmatched line: cos, sin of its world angle (Robot.cpp:794-795) */
};

/* ---- launchers (ekf_kernels.cu); every one is asynchronous on `s` and returns the CUDA status ---- */
cudaError_t ekf_launch_init(const EkfGeom& g, const EkfBuffers& b, cudaStream_t s);
/* carry != NULL: device int, pending terms the scan's sweep group already holds (the scan appends after them) */
cudaError_t ekf_launch_predict(const EkfGeom& g, const EkfBuffers& b, const double* d_u, const double* d_x_t0,
                               int m, int L_ub, cudaStream_t s, const int* carry = 0);
cudaError_t ekf_launch_associate(const EkfGeom& g, const EkfBuffers& b, const double* d_z, const double* d_R,
                                 int line, int L_ub, cudaStream_t s);
/* mode 0: fused slice+gain (single GPU); 1: slice only into colA/colB; 2: gain from colA/colB */
cudaError_t ekf_launch_gain(const EkfGeom& g, const EkfBuffers& b, const double* d_z, const double* d_R,
                            int line, int j_override, int mode, int L_ub, int max_batch, cudaStream_t s);
cudaError_t ekf_launch_apply(const EkfGeom& g, const EkfBuffers& b, int line, int j_override, int L_ub,
                             cudaStream_t s);
int ekf_pick_cluster(void);
void ekf_prefer_max_smem_carveout(void);
/* all lines [line0, line1) of the open scan in one cluster launch (single-GPU path) */
cudaError_t ekf_launch_scan_lines(const EkfGeom& g, const EkfBuffers& b, const double* d_z, const double* d_R,
                                  int line0, int line1, int ctas, int coop, int own_slot0, int prev_slot0,
                                  const int* prev_cnt_ptr, const EkfPeers* peers, int L_ub, cudaStream_t s,
                                  const double* pred_u = 0, const double* pred_x = 0, int pred_m = 0, const int* pred_carry = 0);
/* pred_u != NULL: the scan's prediction (ekf_launch_predict's work for pred_m lines, with pred_carry as its carry) runs as the
 * prologue of this launch; only legal when ekf_scan_lines_fuses_predict(peers) */
int ekf_scan_lines_fuses_predict(const EkfPeers* peers);
cudaError_t ekf_launch_flush_done(const EkfBuffers& b, int next_line, cudaStream_t s);
cudaError_t ekf_launch_chunk_mark(const EkfBuffers& b, int next_line, EkfScanView* view, cudaStream_t s);
cudaError_t ekf_launch_queue_all(const EkfGeom& g, const EkfBuffers& b, int m, cudaStream_t s);
/* np_ptr: device int holding the number of pending terms (NULL = st->np); np_ub: host upper bound (selects the template) */
cudaError_t ekf_launch_sweep(const EkfGeom& g, const EkfBuffers& b, const int* np_ptr, int np_ub, int L_ub,
                             cudaStream_t s);
/* pipelined (TMA + mbarrier) form of the sweep; tmap = CUtensorMap of this rank's P with box (tc, tr) of
 * ekf_sweep_shape(shape); one pass per 8 pending terms */
cudaError_t ekf_launch_sweep_tma(const EkfGeom& g, const EkfBuffers& b, const void* tmap, const void* tmap8, const void* tmapK, const void* tmapKS,
                                 double* dst, int slot0,
                                 const EkfScanView* view, unsigned long long* counters, int shape, int np_ub, int L_ub,
                                 int num_sms, cudaStream_t s, const void* tmap_dst = 0, const void* tmap8_dst = 0);
void ekf_sweep_shape(int shape, int* tr, int* tc);
void ekf_sweep_pbox(int shape, int* rows, int* cols);
int ekf_sweep_terms_per_pass(int shape, int np_ub);
/* P2 != NULL: the new columns are also written there; prev_cnt_ptr != NULL: the appended rows are also zeroed in the
 * *prev_cnt_ptr slots from prev_slot0 (both while a sweep group stays open, DESIGN section 5) */
cudaError_t ekf_launch_end_scan(const EkfGeom& g, const EkfBuffers& b, const double* d_z, const double* d_R,
                                int m, int L_ub, int slot0, EkfScanView* view, cudaStream_t s,
                                double* P2 = 0, int prev_slot0 = 0, const int* prev_cnt_ptr = 0);
cudaError_t ekf_launch_assemble(const EkfGeom& g, const EkfBuffers& b, int r0, int nr, int c0, int nc,
                                double* d_out, int ld_out, cudaStream_t s);
cudaError_t ekf_launch_scatter(const EkfGeom& g, const EkfBuffers& b, int r0, int nr, int nl, const double* d_in,
                               int ld_in, cudaStream_t s);
cudaError_t ekf_launch_cov_stats(const EkfGeom& g, const EkfBuffers& b, double* d_partials, int n_partials,
                                 double* d_out3, cudaStream_t s);
cudaError_t ekf_launch_zero_pending(const EkfGeom& g, const EkfBuffers& b, int m, int* d_np, cudaStream_t s);
/* landmark removal (ekf_remove_lines), keep[i] = old state index of new state index i < nl (strictly increasing).
 * hot: y, rows 0..2 of top and the 2x2 diagonal blocks into stage ((6 nl - 6) doubles, put = 0), then back (put = 1);
 * cold: destination rows [r0, r0 + nr) of the live upper triangle from column max(r, c_from) on; row r lives at
 * dst + (r - dst_row0) * ld_dst and reads source row keep[r] (keep = NULL: row r) at src + (row - src_row0) * ld_src,
 * columns keep[c] (keep = NULL: c).  Single-GPU layout only. */
cudaError_t ekf_launch_remove_hot(const EkfGeom& g, const EkfBuffers& b, const int* keep, int nl, double* stage, int put,
                                  cudaStream_t s);
cudaError_t ekf_launch_remove_cold(const double* src, size_t ld_src, int src_row0, double* dst, size_t ld_dst, int dst_row0,
                                   const int* keep, int r0, int nr, int nl, int c_from, cudaStream_t s);
/* landmark insertion (ekf_insert_lines): k new landmarks L .. L+k-1 appended after the L live ones.
 * hot: src = 5 doubles per new landmark (alfa, r, C[a,a], C[a,b], C[b,b]) -> y (alfa wrapped), zero `top` columns and the
 * 2x2 diagonal blocks; cold: rows [r0, r0 + nr) of the single-GPU P (row stride ld), columns max(r, nl_old) .. nl-1: zeros
 * for r < nl_old, else row r - nl_old of the 2k-wide new block (its row i at blk + (i - blk_row0) * 2k; blk = NULL: zeros). */
cudaError_t ekf_launch_insert_hot(const EkfGeom& g, const EkfBuffers& b, int L, int k, const double* src, cudaStream_t s);
cudaError_t ekf_launch_insert_cold(double* P, size_t ld, int nl_old, int nl, int r0, int nr, const double* blk, int blk_row0,
                                   cudaStream_t s);
/* absolute pose fix (ekf_observe_pose), d = 1..3 selected components, on the complete in-place covariance.
 * gain: S, S^-1, v, d2 and the decision (into st->fix_*), and the gain rows as two rank-2 terms: term 1
 * (K_0, K_1 ; KS_0, KS_1) into pending slot 0, term 2 (K_2, 0 ; KS_2, 0) into (K2, KS2) (slot 1, or a scratch row when
 * there is one slot).  apply: the hot update, y, pose and x_pre, and st->np = the terms the sweep folds (0 when rejected;
 * at most max_np).  term2: copies (K2, KS2) into slot 0 and sets st->np for a second one-term sweep (one slot only). */
cudaError_t ekf_launch_pose_gain(const EkfGeom& g, const EkfBuffers& b, const EkfPoseFix& f, int d, double2* K2,
                                 double2* KS2, int L_ub, cudaStream_t s);
cudaError_t ekf_launch_pose_apply(const EkfGeom& g, const EkfBuffers& b, int d, const double2* K2, const double2* KS2,
                                  int max_np, int L_ub, cudaStream_t s);
cudaError_t ekf_launch_pose_term2(const EkfGeom& g, const EkfBuffers& b, int d, const double2* K2, const double2* KS2,
                                  int L_ub, cudaStream_t s);
int ekf_sweep_grid_ub(const EkfGeom& g, int L_ub);

/* The largest double T with sqrt(T) <= gate (sqrt correctly rounded): Robot.cpp:489's `sqrt(fabs(d2)) > MAHALANOBIS`
 * is then exactly `fabs(d2) > T`, for every d2 including +-inf and NaN (both forms are false for a NaN d2).
 *   gate = +inf or NaN: `sqrt(|d2|) > gate` is false for every d2, so T = +inf (nothing is rejected; the search below
 *                       would never end at +inf, as nextafter(inf, inf) == inf);
 *   gate < 0:           `sqrt(|d2|) > gate` is true for every non-NaN d2, so T = -1 (everything but NaN is rejected). */
#include <math.h>
static inline double ekf_gate_d2max(double gate) {
  if (gate != gate || gate == INFINITY) return INFINITY;
  if (!(gate >= 0.0)) return -1.0;
  double t = gate * gate;
  while (sqrt(t) > gate) t = nextafter(t, 0.0);
  for (;;) { const double u = nextafter(t, INFINITY); if (!(sqrt(u) <= gate)) break; t = u; }
  return t;
}

/* rows of P this rank stores */
static inline int ekf_local_tile_rows(const EkfGeom& g) {
  const int T = g.ld / EKF_TILE;
  return (T - g.rank + g.world - 1) / g.world;
}

#endif
