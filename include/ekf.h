/* ekf.h -- C ABI of libekfcuda: the B200-native EKF-SLAM core behind slam_ros's `Robot`.
 *
 * The reference (HuaiLeiTang/slam_ros) has no FFI: its EKF is ~36 inline gsl_blas_dgemm call sites
 * inside Robot::localize (slam_ros/Robot.cpp:126-943).  This header is the boundary a maintainer
 * binds instead of those calls (INTEGRATION.md shows the Robot.cpp replacement).  Each entry point
 * cites the reference lines it replaces.  Conventions:
 *
 *   - plain C, plain pointers and sizes; all pointers are HOST pointers unless the name says _device;
 *   - every function returns an int status (EKF_OK == 0), mirroring the reference's "collect the GSL
 *     int code, never abort" convention (Robot.cpp:240-261, 909-913);
 *   - one ekf_ctx per Robot, NOT thread-safe (the node is single-threaded: slam_ros/main.cpp:130-178),
 *     one CUDA stream per ctx;
 *   - state layout is the reference's (Robot.h:26-28, 62):  y = [x, y, theta, alfa_0, r_0, alfa_1, ...],
 *     a line is (alfa, r) -- ANGLE FIRST (simplifyPath.h:62-79) -- with R = its 2x2 C_AR, row-major;
 *   - the covariance stays resident in HBM across calls.  On the device only the UPPER triangle is
 *     authoritative (the reference's P drifts asymmetric at the ulp level -- Robot.cpp:568 is a
 *     full-matrix, non-symmetrised update); downloads are symmetrised.
 *   - there is no CPU fallback: without a CUDA device ekf_create fails with EKF_ECUDA.
 */
#ifndef LIBEKFCUDA_EKF_H
#define LIBEKFCUDA_EKF_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ekf_ctx ekf_ctx;

enum {
  EKF_OK = 0,
  EKF_EINVAL = 1,     /* bad argument */
  EKF_ECAPACITY = 2,  /* a new line did not fit (the reference overruns y[] here -- SURVEY Q4); line dropped */
  EKF_ESINGULAR = 3,  /* innovation covariance S singular for some pair; pair treated as "no match" */
  EKF_ECUDA = 4,      /* CUDA runtime failure (message: ekf_last_error) */
  EKF_ENCCL = 5,      /* NCCL failure in the row-sharded mode */
  EKF_ENOMEM = 6,
  EKF_ESTATE = 7      /* call out of sequence (e.g. ekf_update before ekf_predict) */
};

enum {
  EKF_FLAG_EAGER_SWEEP = 1,  /* sweep P after every matched line (one rank-2 pass per match, like the
                                reference) instead of folding the scan's matches into one rank-2m pass */
  EKF_FLAG_PER_LINE_KERNELS = 4, /* ekf_scan launches associate / gain / apply per line instead of the single
                                    cluster kernel that walks all lines (same bits; A/B measurement) */
  EKF_FLAG_NO_OVERLAP = 8,   /* do not double-buffer P / overlap a scan's sweep with the next scan's line loop */
  EKF_FLAG_SWEEP_DIRECT = 2, /* use the plain load/compute/store sweep kernel instead of the TMA + mbarrier
                                pipeline (same bits; kept for A/B measurement) */
  EKF_FLAG_FULL_GATES = 16   /* evaluate the full Mahalanobis gate (Robot.cpp:367-489) for EVERY landmark instead of
                                first discarding those whose angle innovation alone puts them beyond twice the gate
                                (d^2 >= v0^2 / S00); same associations, kept for A/B measurement and as a test */
};

typedef struct {
  int capacity_lines;   /* LINESIZE            (Robot.h:13, 100)   */
  double gate;          /* MAHALANOBIS         (Robot.h:15, 0.4)   */
  double encoder_noise; /* ENCODERNOISE        (Robot.h:17, 0.024) */
  int reset_headroom;   /* the 10 of "savedLineCount > LINESIZE-10" (Robot.cpp:893) */
  int device;           /* CUDA device ordinal */
  int max_batch;        /* most lines folded into one deferred in-place sweep (default 64; <= 0 means 64).  It counts
                           lines on the scan paths (matched or not) and ekf_update calls on the step-wise path.  It also
                           sizes the overlapped pipeline: below 16 nothing overlaps; from 16 to 63 the slot ring halves
                           hold max_batch / 2 (at most 32) terms, and scans of more lines than that, up to 32, run in
                           place; from 64 on they hold 64.  Above 64 the fused line loop is off: in-place scans run the
                           per-line kernels.  Every value gives the same results, bit for bit. */
  int flags;            /* EKF_FLAG_* */
} ekf_config;

/* Fills the reference's compile-time constants (Robot.h:13-17). */
int ekf_default_config(ekf_config* cfg);

/* Robot::Robot (Robot.cpp:20-35): zero-filled y and P, P[0,0] = P[1,1] = 0.05, pose = 0. */
int ekf_create(ekf_ctx** out, const ekf_config* cfg);
int ekf_destroy(ekf_ctx* ctx);
const char* ekf_last_error(const ekf_ctx* ctx);

/* --- the step-wise path: one call per reference block -------------------------------------------
 * A step-wise scan (ekf_predict ... ekf_end_scan) holds at most 64 lines -- more once a fused ekf_scan with more
 * lines has run on the ctx (its line tables only grow between scans); a 65th ekf_associate / ekf_update /
 * ekf_add_line returns EKF_EINVAL and leaves the scan open.  The fused ekf_scan has no such limit. */

/* Robot.cpp:130-258: x_pre = f(x_t0, u); P <- Fx P Fx' + Fu Q Fu'.  Starts a scan (clears the
 * per-scan match list, Robot.cpp:288-295).  x_t0 == NULL uses the resident pose (xPos,yPos,thetaPos).
 * u = (translation, unused, rotation) as built at Robot.cpp:135-145.  x_pre (nullable) gets the 3 doubles. */
int ekf_predict(ekf_ctx* ctx, const double x_t0[3], const double u[3], double x_pre[3]);

/* Robot.cpp:298-501 for ONE observed line against every not-yet-matched landmark: innovation,
 * S = H P H' + R, LU inverse, Mahalanobis gate, FIRST-FIT (lowest index that passes -- the reference
 * `break`s at :641).  *j_out = landmark index or -1.  innov (nullable) = (z - h) after the wraps. */
int ekf_associate(ekf_ctx* ctx, const double z[2], const double R[4], int* j_out, double innov[2]);

/* Robot.cpp:516-602 for landmark j: K = P H' S^-1, P -= (K S) K', y += K (z - h), pose mirrors.
 * x_post (nullable) = the updated robot pose. */
int ekf_update(ekf_ctx* ctx, int j, const double z[2], const double R[4], double x_post[3]);

/* extraLines.push_back (Robot.cpp:309, 325, 493): queue an unmatched line; it is appended to the
 * state by ekf_end_scan in queue order (Robot.cpp:776-866). */
int ekf_add_line(ekf_ctx* ctx, const double z[2], const double R[4]);

/* Robot.cpp:702-716 (no-line / no-match pose), :776-866 (augmentation of the queued lines),
 * :893-904 (map reset when savedLineCount > capacity - headroom).  Flushes the deferred sweep.
 * pose (nullable) = xPos, yPos, thetaPos. */
int ekf_end_scan(ekf_ctx* ctx, int n_lines, double pose[3]);

/* --- the fused path ----------------------------------------------------------------------------- */

/* One whole Robot::localize: predict, then for each of the m lines (in order) associate / update or
 * queue, then end-of-scan.  Nothing returns to the host between lines; the scan's matched updates are
 * folded into one rank-2m sweep of P.  z = m x (alfa, r), R = m x 4.  j_out (nullable, m ints) = matched
 * landmark or -1 per line.  pose (nullable) = resulting xPos, yPos, thetaPos. */
int ekf_scan(ekf_ctx* ctx, const double x_t0[3], const double u[3], int m, const double* z,
             const double* R, int* j_out, double pose[3]);

/* Same, asynchronous, with DEVICE-resident inputs (d_u: 3, d_z: 2m, d_R: 4m doubles) and a device
 * output d_j_out (nullable, m ints).  Uses the resident pose as x_t0.  Returns after enqueueing. */
int ekf_scan_device(ekf_ctx* ctx, const double* d_u, int m, const double* d_z, const double* d_R,
                    int* d_j_out);
int ekf_sync(ekf_ctx* ctx);

/* --- state access -------------------------------------------------------------------------------- */

/* xPos/yPos/thetaPos, savedLineCount and the sticky status (EKF_ECAPACITY / EKF_ESINGULAR seen since
 * the last call; cleared by the call).  Any pointer may be NULL.
 *
 * Status of a scan.  EKF_ECAPACITY: more unmatched lines than free slots; the first ones in line order were appended,
 * the rest dropped (then the reset policy applies as usual).  EKF_ESINGULAR: the first fit of some line skipped a
 * pair whose S has a zero pivot in its LU before the landmark it matched (or anywhere, if it matched nothing); the
 * search went on past it.  A singular pair past a line's match is not reported, on any path.  When a scan hits both,
 * EKF_ECAPACITY is reported.
 * Every scan ORs its status into a sticky word on the device.  ekf_scan and ekf_end_scan return it and clear it, so
 * they report their own scan plus any ekf_scan_device scan not read yet, and the next clean scan returns EKF_OK.
 * ekf_scan_device reports nothing: ekf_get_state with sticky_status != NULL waits for the scans enqueued before it,
 * returns the word (ECAPACITY first) and clears it; with sticky_status == NULL it leaves the word as it is. */
int ekf_get_state(ekf_ctx* ctx, double pose[3], int* n_lines, int* sticky_status);

/* P_t0[0:3,0:3] row-major, symmetrised: what Robot::getEllipse reads (Robot.cpp:75-77). */
int ekf_get_robot_cov(ekf_ctx* ctx, double Prr[9]);

/* Robot::getEllipse (Robot.cpp:73-124) in closed form: axii = 2*sqrt(5.991*|lambda|) ascending in
 * |lambda|; angle = atan2(v_x, v_y) of the major eigenvector.  Returns EKF_OK, *ok = 1 on success. */
int ekf_get_ellipse(ekf_ctx* ctx, float axii[2], float* angle, int* ok);

/* Whole state in the reference's own layout: y[n], P[n*n] row-major with n = 3 + 2*capacity_lines,
 * zeros outside the live part (this is Robot::y / Robot::P_t0).  Either pointer may be NULL. */
int ekf_download(ekf_ctx* ctx, double* y, double* P, int* n_lines);
int ekf_upload(ekf_ctx* ctx, const double* y, const double* P, int n_lines);

/* Map management, not in the reference.  Removes landmarks lines[0..k) (strictly increasing, each in
 * [0, savedLineCount)) from the map: their entries of y and their rows and columns of P are deleted and the later
 * landmarks move down in order (landmark j becomes j minus the number of removed indices below it) -- the marginal of
 * the remaining state, pure data movement, bit for bit.  Waits for the sweep in flight.  *n_lines (nullable) = the new
 * savedLineCount.  k = 0 is a no-op.  The caller chooses the indices (ekf_scan's j_out says which landmarks each scan
 * matched); the library has no removal policy of its own, and the map reset of Robot.cpp:893-904 is unchanged.
 * EKF_EINVAL: bad list (unsorted, duplicate, out of range, k < 0, NULL with k > 0), or a row-sharded filter (rows would
 * move between ranks); EKF_ESTATE: inside an open step-wise scan.  On error the state is unchanged.  The Monte-Carlo
 * batch filters (ekf_batch_*) have no such call. */
int ekf_remove_lines(ekf_ctx* ctx, int k, const int* lines, int* n_lines);

/* Map management, not in the reference.  Appends k known landmarks -- the walls of a floor plan, or the map of an earlier
 * session -- as landmarks savedLineCount .. savedLineCount+k-1, in order.  lines = k x (alfa, r) in the world frame, the
 * convention of the state's own landmarks y[3+2j], y[4+2j]; alfa is stored after normalize_radian (Robot.cpp:62-71) as
 * the augmentation stores it (:801), r as given.  cov = NULL: surveyed, every new entry of P is zero; otherwise the
 * 2k x 2k row-major joint covariance of the new landmarks (for example the landmark block P[3:, 3:] of an earlier
 * session's ekf_download_live).  The cross-covariance with the robot and the existing landmarks is zero.  The result is
 * bit for bit y' = [y, lines], P' = [[P, 0], [0, cov]]; pose, x_pre and the robot covariance are unchanged.  Waits for
 * the sweep in flight.  *n_lines (nullable) = the new savedLineCount.  k = 0 is a no-op.
 * A landmark with zero covariance stays fixed under every scan: its rows of P are zero, so its gain rows are zero, and a
 * line that matches it is a pure pose measurement.  One with a prior covariance is an ordinary landmark from then on.
 * First fit takes the lowest landmark index, so a floor plan wins over SLAM duplicates of its walls only if it is
 * inserted on a fresh filter before the first scan, or after the duplicates are removed (ekf_remove_lines).
 * The map reset of Robot.cpp:893-904 counts inserted landmarks like any others and drops them with the map; a caller
 * that wants them kept re-inserts them after a reset, which it sees as the line count falling.
 * EKF_EINVAL: k < 0, NULL lines with k > 0, a non-finite entry, a cov that is not exactly symmetric, has a non-finite
 * entry or a negative diagonal entry (positive semi-definiteness beyond that is not checked: it would cost O(k^3)), or a
 * row-sharded filter; EKF_ECAPACITY: savedLineCount + k > capacity_lines -- the call is all or nothing, unlike a scan's
 * augmentation, which appends what fits; EKF_ESTATE: inside an open step-wise scan.  On error the state is unchanged.
 * The Monte-Carlo batch filters (ekf_batch_*) have no such call.
 * Cost (one B200, DESIGN section 3.3): writes 8 (nl_old 2k + k (2k + 1)) bytes of P at about the device-to-device copy
 * rate plus a fixed cost: 100 surveyed walls into 10 000 landmarks 0.05 ms; with cov, the host-side check and the
 * pageable copy of cov dominate (5.1 ms for k = 1 000). */
int ekf_insert_lines(ekf_ctx* ctx, int k, const double* lines, const double* cov, int* n_lines);

/* Absolute pose measurement, not in the reference (GNSS, UWB, motion capture, a docking fiducial, a relocaliser).
 * mask selects d = popcount(mask) components of the pose; z is a full 3-vector (x, y, theta) and R a full row-major 3x3
 * covariance, of which only the selected entries are read.  With H = the selected rows of [I_3 0]:
 *   v = z_sel - y_sel (the theta component wrapped by normalize_radian, Robot.cpp:62-71), S = H P H' + R_sel (from the
 *   upper triangle), S^-1 by LU with partial pivoting, d2 = v' S^-1 v, K = P H' S^-1, P -= (K S) K', y += K v, then
 *   normalize_radian(y[2]); the pose (xPos, yPos, thetaPos) and x_pre follow y[0:3], as after a line update
 *   (Robot.cpp:516-602 with d x d blocks).
 * The fix is accepted iff S is nonsingular and d2 <= d2_max (a chi-square threshold for d degrees of freedom; +inf
 * accepts everything, a NaN d2 is rejected).  A rejected fix leaves the state bit for bit unchanged and returns EKF_OK
 * with *accepted = 0; a singular S (e.g. theta alone on a fresh filter, P[2,2] = 0, with R_thth = 0) returns
 * EKF_ESINGULAR, state unchanged.  d2, accepted and pose (the resulting xPos, yPos, thetaPos) are nullable; when all three
 * are NULL the call returns after enqueueing and a singular S is not reported.  Waits for the sweep in flight.
 * EKF_EINVAL: mask 0 or above 7, NULL z or R, a non-finite selected entry, a selected R that is not symmetric, a NaN
 * d2_max, or a row-sharded filter; EKF_ESTATE: inside an open step-wise scan.  On error the state is unchanged.  The
 * Monte-Carlo batch filters (ekf_batch_*) have no such call. */
enum { EKF_POSE_X = 1, EKF_POSE_Y = 2, EKF_POSE_THETA = 4 };
int ekf_observe_pose(ekf_ctx* ctx, int mask, const double z[3], const double R[9], double d2_max, double* d2,
                     int* accepted, double pose[3]);

/* Live part only: nl = 3 + 2*savedLineCount entries of y and an nl x nl block with row stride ldp.
 * Fails with EKF_EINVAL if nl > max_n. */
int ekf_download_live(ekf_ctx* ctx, double* y, double* P, int ldp, int max_n, int* n_lines);
/* An nr x nc block of the (symmetrised) covariance starting at (r0, c0); row stride nc. */
int ekf_download_block(ekf_ctx* ctx, int r0, int c0, int nr, int nc, double* out);
/* Size-independent invariants for full-size checks: trace, sum and sum of squares of the live,
 * symmetrised covariance (device reductions in fixed order: deterministic). */
int ekf_cov_stats(ekf_ctx* ctx, double* trace, double* sum, double* sumsq);

/* --- measurement --------------------------------------------------------------------------------- */

/* CUDA-event accounting on the ctx stream.  While enabled, every covariance sweep is bracketed by
 * events; ekf_profile_read returns the number of sweeps, their total device time and the algorithmic
 * bytes they moved (8 n (n+1) + 32 n m per sweep, SURVEY 8d), then resets the counters.
 * launches = kernels launched by this ctx since the last read. */
int ekf_profile_enable(ekf_ctx* ctx, int on);
int ekf_profile_read(ekf_ctx* ctx, int* n_sweeps, double* sweep_ms, double* sweep_bytes, long long* launches);
/* Same accounting for the OTHER half of a scan: device time between the start of the prediction and the end of
 * the line loop (overlapped scans: the end of the augmentation kernels) -- i.e. how long the line stream is busy
 * per scan, the quantity the sweep has to hide.  Call before ekf_profile_read (which leaves profiling on). */
int ekf_profile_read_lines(ekf_ctx* ctx, int* n_scans, double* line_ms);

/* Device-time bracket on the ctx stream (CUDA events): start records an event, stop records a second
 * one, waits for it and returns the elapsed milliseconds.  This is how bench.py times K steps. */
int ekf_timer_start(ekf_ctx* ctx);
int ekf_timer_stop(ekf_ctx* ctx, double* ms);

/* Stand-alone covariance sweep for the roofline measurement: applies `m` synthetic rank-2 terms
 * (K = KS = 0, so P is unchanged bit for bit) over the live part; reports device ms via events. */
int ekf_sweep_probe(ekf_ctx* ctx, int m, int repeats, double* ms_each);

/* --- row-sharded covariance across GPUs (one process per GPU) -------------------------------------
 * Rank `rank` of `world` owns the 64-row tile rows rb with rb % world == rank of the SAME filter; y,
 * rows 0-2 and the 2x2 diagonal blocks are replicated.  Per matched line the ranks exchange the two
 * H-column slices (16 n bytes) with NCCL.  nccl_unique_id: the 128 bytes of ncclGetUniqueId made by
 * rank 0 (ekf_nccl_unique_id) and distributed by the host (e.g. torch.distributed broadcast). */
int ekf_nccl_unique_id(unsigned char id[128]);
int ekf_create_sharded(ekf_ctx** out, const ekf_config* cfg, int rank, int world,
                       const unsigned char nccl_unique_id[128]);

/* Fused exchange: after ekf_shard_connect + ekf_shard_use_fused(1) the H-column slices no longer go through NCCL.  The line-loop kernel
 * itself stores the slice entries a rank owns straight into every peer's exchange buffer over NVLink (peer memory
 * mapped with CUDA IPC), publishes an arrival epoch with a system-scope release store and spins (bounded) on its
 * own flags -- one NVLink round trip per matched line, no kernel boundary, and the scan's sweep then overlaps
 * the next scan's line loop exactly as on one GPU.  ekf_shard_ipc_handle returns the 64-byte cudaIpcMemHandle_t
 * of this rank's buffer; the host all-gathers the handles (rank order, world x 64 bytes) and hands them to
 * ekf_shard_connect on every rank.  world <= 8 (one NVSwitch domain).  If a peer cannot be mapped the call
 * returns EKF_ECUDA and the filter stays on the NCCL exchange.  A peer that never arrives makes the scan return
 * EKF_ENCCL instead of hanging the GPU. */
int ekf_shard_ipc_handle(ekf_ctx* ctx, unsigned char handle[64]);
int ekf_shard_connect(ekf_ctx* ctx, const unsigned char* handles);
/* Two-phase switch: ekf_shard_connect only MAPS the peers; the ranks then agree (host-side, e.g. an all-reduce
 * MIN of the outcomes) and every rank calls ekf_shard_use_fused(ctx, all_mapped) -- ranks on different exchange
 * paths would wait for each other forever.  on = 0 returns to the NCCL exchange. */
int ekf_shard_use_fused(ekf_ctx* ctx, int on);

/* --- independent filters (Monte-Carlo batch): no communication -------------------------------------
 * B filters of identical capacity on one device, one thread block per filter, covariance staged in
 * shared memory for the whole scan. */
typedef struct ekf_batch ekf_batch;
int ekf_batch_create(ekf_batch** out, const ekf_config* cfg, int n_filters);
int ekf_batch_destroy(ekf_batch* b);
/* One localize per filter.  u: B x 3, z: B x m x 2, R: B x m x 4, j_out (nullable): B x m, pose (nullable): B x 3.
 * Status: of this step alone, over all filters: EKF_ECAPACITY if a filter dropped a line, else EKF_ESINGULAR if a
 * filter's first fit skipped a singular pair before its match (as for ekf_get_state).  One exception: without
 * EKF_FLAG_FULL_GATES a landmark with S00 > 0 whose angle innovation alone puts it beyond twice the gate is not gated
 * in full, so a singular S of that pair goes unreported (the association is the same: it is no match either way); a
 * pair with S00 == 0 is always gated. */
int ekf_batch_scan(ekf_batch* b, const double* u, int m, const double* z, const double* R, int* j_out,
                   double* pose);
/* The same, pipelined: ekf_batch_submit stages the step's inputs and returns at once (at most two steps in flight: the
 * inputs of step s+1 are copied while the kernel of step s runs); ekf_batch_collect waits for the OLDEST submitted step
 * and returns its matches, poses and status: the status of that step, not of the one submitted after it.
 * ekf_batch_scan == submit + collect.  ekf_batch_scan_device reports no status. */
int ekf_batch_submit(ekf_batch* b, const double* u, int m, const double* z, const double* R);
int ekf_batch_collect(ekf_batch* b, int* j_out, double* pose);
int ekf_batch_scan_device(ekf_batch* b, const double* d_u, int m, const double* d_z, const double* d_R,
                          int* d_j_out);
int ekf_batch_sync(ekf_batch* b);
int ekf_batch_download(ekf_batch* b, int filter, double* y, double* P, int* n_lines, double pose[3]);
const char* ekf_batch_last_error(const ekf_batch* b);

/* --- line extraction on the device (SURVEY 8f row 2) -------------------------------------------------
 * What the node does with one `mappingPoints` payload before Robot::localize: slam_ros/main.cpp:37-71
 * (`mapping_cb`: (r, angle) float pairs, alfa = angle - pi, returns with r > 0.05 m, variance 0.01) and
 * LineExtraction (slam_ros/lineFitting.cpp:640-702: sort, 0.5 m segmentation, recursive split, fit, finite-
 * difference covariance, end points, LineConversion), then alfa += pi (main.cpp:66-69).  Output per line, in the
 * reference's order: 10 doubles = alfa, r, C_AR[4] (row-major, off-diagonals 0), lineInterval[0] (alfa, r),
 * lineInterval[1] (alfa, r) -- i.e. the `line` fields Robot::localize reads (simplifyPath.h:62-79).
 * At most 4096 points per payload.  *n_lines may exceed max_lines (then only max_lines were written). */
typedef struct ekf_lx ekf_lx;
int ekf_lx_create(ekf_lx** out, int device, int max_lines);
int ekf_lx_destroy(ekf_lx* lx);
const char* ekf_lx_last_error(const ekf_lx* lx);
int ekf_lx_extract(ekf_lx* lx, int n_pairs, const float* data, int* n_lines, double* lines);
/* Asynchronous, payload already in HBM; the results stay there in the layout ekf_scan_device consumes:
 * *d_z = max_lines x (alfa, r), *d_R = max_lines x 4, *d_count = the number of lines (device int). */
int ekf_lx_extract_device(ekf_lx* lx, int n_pairs, const float* d_data, const double** d_z, const double** d_R,
                          const int** d_count);
int ekf_lx_sync(ekf_lx* lx);
/* The consumers after the filter (SURVEY 8f row 4).  lineprovider/main.cpp:60-84 (Transform): the two end points of every
 * line of the LAST extraction, from the robot frame to the world frame with the filter's pose (x, y, theta) -- what the
 * `lines_1` topic carries, 4 floats (x0, y0, x1, y1) per line; astar/main.cpp:44-73 (lines_cb) takes those floats times
 * 100 as the planner's obstacle segments in centimetres: scale = 100 (a float product, as there), scale = 1 for `lines_1`
 * itself.  *n_lines = lines of the last extraction; at most max_out_lines are written. */
int ekf_lx_world_segments(ekf_lx* lx, const double pose[3], double scale, float* out, int max_out_lines, int* n_lines);

const char* ekf_version(void);

#ifdef __cplusplus
}
#endif
#endif
