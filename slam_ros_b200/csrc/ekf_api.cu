/* ekf_api.cu -- the extern "C" boundary of libekfcuda (include/ekf.h): context, HBM residency,
 * stream ordering, the per-scan launch sequence, measurement taps and the NCCL exchange of the
 * row-sharded mode.  No arithmetic of the filter lives here -- it is all in ekf_kernels.cu.
 */
#include "../../include/ekf.h"
#include "ekf_internal.h"

#include <cuda.h>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

/* ---- NCCL, bound at run time so that the library shares whatever libnccl the host process already
 *      loaded (torch bundles its own) and has no link-time dependency in the single-GPU case ---- */
namespace {
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
struct NcclApi {
  void* handle;
  int (*GetUniqueId)(ncclUniqueId*);
  int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
  int (*CommDestroy)(ncclComm_t);
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t);
  const char* (*GetErrorString)(int);
};
const int kNcclFloat64 = 8, kNcclSum = 0;

NcclApi* nccl_api() {
  static NcclApi api = {0, 0, 0, 0, 0, 0};
  static int tried = 0;
  if (!tried) {
    tried = 1;
    const char* names[] = {"libnccl.so.2", "libnccl.so", 0};
    for (int i = 0; names[i] && !api.handle; ++i) api.handle = dlopen(names[i], RTLD_NOW | RTLD_GLOBAL);
    if (api.handle) {
      api.GetUniqueId = (int (*)(ncclUniqueId*))dlsym(api.handle, "ncclGetUniqueId");
      api.CommInitRank = (int (*)(ncclComm_t*, int, ncclUniqueId, int))dlsym(api.handle, "ncclCommInitRank");
      api.CommDestroy = (int (*)(ncclComm_t))dlsym(api.handle, "ncclCommDestroy");
      api.AllReduce = (int (*)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t))dlsym(api.handle, "ncclAllReduce");
      api.GetErrorString = (const char* (*)(int))dlsym(api.handle, "ncclGetErrorString");
      if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllReduce) api.handle = 0;
    }
  }
  return api.handle ? &api : 0;
}
}  // namespace

struct ekf_ctx {
  ekf_config cfg;
  EkfGeom g;
  EkfBuffers b;
  cudaStream_t stream;
  /* per-scan inputs owned by the ctx (host path and step-wise path) */
  int max_lines;
  double* d_in;        /* [u(3) | x_t0(3) | z(2*max_lines) | R(4*max_lines)] */
  double* h_in;        /* pinned mirror */
  int* h_jout;         /* pinned */
  EkfDevState* h_st;   /* pinned */
  /* device-resident scans never wait for the GPU, so the host only knows an upper bound of the map size (it sizes grids and
   * picks the line-loop form).  A snapshot of the device state is copied back asynchronously now and then; once it has
   * landed, the bound restarts from the snapshot plus the lines enqueued after it. */
  EkfDevState* h_snap; /* pinned */
  cudaEvent_t ev_snap;
  int snap_inflight, snap_added;
  /* host-side view of the device state */
  int L_ub;            /* upper bound of savedLineCount */
  int pend_ub;         /* upper bound of the pending-term count */
  int scan_open;
  int cursor;          /* lines consumed by the open step-wise scan */
  /* measurement */
  int prof;
  std::vector<cudaEvent_t> ev;
  size_t ev_used;
  std::vector<double> ev_bytes;
  std::vector<cudaEvent_t> lev;   /* event pairs around the line-stream part of each scan (predict .. line loop [.. end of scan]) */
  size_t lev_used;
  long long launches;
  cudaEvent_t t0, t1;  /* ekf_timer_* */
  /* overlapped pipeline: the sweep of scan s runs on `wstream` while scan s+1's line loop runs on `stream`.
   * P is double-buffered; a sweep reads Pbuf[x] and writes Pbuf[x^1].  `rd` is the buffer the line loop
   * reads; `pg_*` describe the previous scan's pending terms that are not folded into Pbuf[rd] yet. */
  int overlap;
  cudaStream_t wstream;
  double* Pbuf[2];
  CUtensorMap tmap2[2];
  CUtensorMap tmap8[2];        /* the same buffers as 64-row x 8-column boxes (tensor-core sweep, k_sweep_dmma) */
  int have_tmap8;
  CUtensorMap tmapK[2];        /* [0]: K bands (box = tile columns x 8 slots), [1]: K S bands (box = tile rows x 8 slots) */
  int rd, par, group;
  int tabpar;                  /* per-line table set of the next overlapped scan */
  int last_line_sms;           /* SMs the most recent sweep launch left free for the line loop */
  int no_fuse;                 /* EKF_FUSE_PREDICT=0: the prediction stays a launch of its own (A/B) */
  void* arena; size_t arena_bytes;   /* y | top | diag | gates | matched | colA,colB | Kp | KSp (one allocation: one L2 window) */
  int chunk_lines, chunk_above;/* overlapped scans of more than chunk_above lines run as chunks of chunk_lines (EKF_CHUNK, EKF_CHUNK_ABOVE; 0 = never) */
  int slots;                   /* rows of Kp / KSp: max(max_batch, 2 * group) */
  int pg_valid, pg_slot0;
  /* sweep groups: consecutive overlapped scans whose pending terms share ONE sweep pass (DESIGN section 5).  At most one
   * group is open; its terms live in half `par` of the slot ring and its sweep is launched when it closes. */
  int grp_budget;              /* most terms a group may hold (EKF_SWEEP_GROUP; 0 = one sweep per scan) */
  int grp_open, grp_terms;     /* grp_terms: upper bound of the open group's terms (the sum of its scans' m) */
  int grp_line_sms;            /* SMs of its scans' line loops (one class per group) */
  int grp_may_reset;           /* one of its scans may have reset the map */
  EkfScanView* d_view;        /* [2] */
  unsigned long long* d_counters;   /* tile counters of the sweep passes: [0,16) line stream, [16,32) sweep stream */
  cudaEvent_t evE, evF[2];
  int evF_used[2];
  struct { int *jbest, *jsing, *jout, *pidx, *eidx, *ext; double* ext_cs; } tab[2];
  int num_sms;
  int cluster;         /* CTAs in the line-loop cluster */
  int sweep_shape;     /* 0: 64x64 tiles, 1: 32x128, 2: 16x256 (EKF_SWEEP_SHAPE) */
  /* sharded */
  ncclComm_t comm;
  double* xchg;               /* this rank's exchange buffer: [2 halves][colA | colB][ld] doubles + 8 arrival flags */
  void* peer_map[8];          /* the peers' buffers as mapped by cudaIpcOpenMemHandle (NULL for the local one) */
  EkfPeers peers;
  int peers_mapped;           /* ekf_shard_connect succeeded: every peer's exchange buffer is mapped */
  int peers_ok;               /* ekf_shard_use_fused(1): the H-column slices travel inside the line-loop kernel */
  int poisoned;               /* a cross-GPU exchange timed out (EKF_ENCCL): the replicas may have diverged; every call
                                 fails with EKF_ESTATE until ekf_upload restores a complete state */
  /* staging for download / upload / stats */
  double* d_stage; size_t stage_elems;
  double* d_partials; double* d_out3;
  int* d_keep;                /* ekf_remove_lines: old state index of every kept one (n ints, allocated on first use) */
  char err[256];
};

namespace {

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) {                                                                  \
      snprintf(ctx->err, sizeof ctx->err, "%s:%d %.120s: %s", "ekf_api.cu", __LINE__, #call, cudaGetErrorString(e_)); \
      return EKF_ECUDA;                                                                       \
    }                                                                                         \
  } while (0)

#define NOT_POISONED(ctx)                                                                                          \
  do {                                                                                                             \
    if ((ctx)->poisoned) {                                                                                         \
      snprintf((ctx)->err, sizeof (ctx)->err, "a cross-GPU exchange timed out earlier (EKF_ENCCL): re-upload the state with ekf_upload"); \
      return EKF_ESTATE;                                                                                           \
    }                                                                                                              \
  } while (0)

const size_t kStageElems = (size_t)8 << 20;   /* 64 MiB staging for download/upload */
const int kOverlapMinN = 6000;                /* below this state dimension the synchronous path is used */
/* SMs reserved for the line loop while a sweep is in flight.  The line loop's time is inversely proportional to
 * its SM count (measured, 10k and 40k landmarks), the sweep's grows only with the SMs it loses; 20 balances the
 * two on one GPU at 10k landmarks.  A row-sharded filter sweeps 1/world of the triangle but still walks every
 * landmark and every row per line, so there the line loop gets more (28 from 4 ranks up). */
static int line_sms_env() { static int v = -2; if (v == -2) { const char* e = getenv("EKF_LINE_SMS"); v = e ? atoi(e) : -1; if (v < 1 || v > 64) v = -1; } return v; }
/* Single GPU: when a few more SMs give the line loop one thread per landmark of the CAPACITY (up to 28 SMs = 14 336 lines),
 * it takes them: the form that keeps a thread's landmark in registers is then valid whatever the map has grown to, also in
 * long device-resident bursts where the host only has a drifting upper bound of the map size. */
static int line_sms_for(int world, int cap, int m) {
  const int e = line_sms_env();
  if (e > 0) return e;
  if (world >= 4) return 28;
  const int need = (cap + 511) / 512;
  /* up to 8 lines per scan the step is bound by the sweep, which keeps the two SMs (0.7 % of the step at 10k landmarks) */
  return (world == 1 && m > 8 && need > 20 && need <= 28) ? need : 20;
}

double* in_u(ekf_ctx* c) { return c->d_in; }
double* in_x(ekf_ctx* c) { return c->d_in + 3; }
double* in_z(ekf_ctx* c) { return c->d_in + 6; }
double* in_R(ekf_ctx* c) { return c->d_in + 6 + 2 * (size_t)c->max_lines; }

void use_tables(ekf_ctx* ctx, int t) {
  ctx->b.jbest = ctx->tab[t].jbest; ctx->b.jsing = ctx->tab[t].jsing; ctx->b.jout = ctx->tab[t].jout; ctx->b.pidx = ctx->tab[t].pidx;
  ctx->b.eidx = ctx->tab[t].eidx; ctx->b.ext = ctx->tab[t].ext; ctx->b.ext_cs = ctx->tab[t].ext_cs;
}

int free_line_tables(ekf_ctx* ctx) {
  for (int t = 0; t < 2; ++t) {
    cudaFree(ctx->tab[t].jbest); cudaFree(ctx->tab[t].jsing); cudaFree(ctx->tab[t].jout); cudaFree(ctx->tab[t].pidx); cudaFree(ctx->tab[t].eidx);
    cudaFree(ctx->tab[t].ext); cudaFree(ctx->tab[t].ext_cs);
    memset(&ctx->tab[t], 0, sizeof ctx->tab[t]);
  }
  cudaFree(ctx->d_in);
  cudaFreeHost(ctx->h_in); cudaFreeHost(ctx->h_jout);
  ctx->b.jbest = ctx->b.jsing = ctx->b.jout = ctx->b.pidx = ctx->b.eidx = ctx->b.ext = 0; ctx->b.ext_cs = 0; ctx->d_in = 0;
  ctx->h_in = 0; ctx->h_jout = 0;
  return 0;
}

int drain(ekf_ctx* ctx);
int close_group(ekf_ctx* ctx);

/* (re)allocate everything sized by the number of lines in a scan; only legal between scans */
int ensure_lines(ekf_ctx* ctx, int m) {
  if (m <= ctx->max_lines) return EKF_OK;
  if (ctx->scan_open && ctx->cursor > 0) {
    snprintf(ctx->err, sizeof ctx->err, "scan has more than %d lines; raise it by calling ekf_scan once with m lines", ctx->max_lines);
    return EKF_EINVAL;
  }
  { int rc = drain(ctx); if (rc) return rc; }
  CU(cudaStreamSynchronize(ctx->stream));
  free_line_tables(ctx);
  int cap = ctx->max_lines > 0 ? ctx->max_lines : 64;
  while (cap < m) cap *= 2;
  ctx->max_lines = 0;             /* committed only once every table below exists: a failed allocation sends the next call back here */
  const size_t n1 = (size_t)cap + 1;
  for (int t = 0; t < 2; ++t) {
    CU(cudaMalloc(&ctx->tab[t].jbest, n1 * sizeof(int)));
    CU(cudaMalloc(&ctx->tab[t].jsing, n1 * sizeof(int)));
    CU(cudaMalloc(&ctx->tab[t].jout, n1 * sizeof(int)));
    CU(cudaMalloc(&ctx->tab[t].pidx, n1 * sizeof(int)));
    CU(cudaMalloc(&ctx->tab[t].eidx, n1 * sizeof(int)));
    CU(cudaMalloc(&ctx->tab[t].ext, n1 * sizeof(int)));
    CU(cudaMalloc(&ctx->tab[t].ext_cs, 2 * n1 * sizeof(double)));
    CU(cudaMemsetAsync(ctx->tab[t].pidx, 0, n1 * sizeof(int), ctx->stream));
    CU(cudaMemsetAsync(ctx->tab[t].eidx, 0, n1 * sizeof(int), ctx->stream));
  }
  use_tables(ctx, 0);
  CU(cudaMalloc(&ctx->d_in, (6 + 6 * (size_t)cap) * sizeof(double)));
  CU(cudaMallocHost(&ctx->h_in, (6 + 6 * (size_t)cap) * sizeof(double)));
  CU(cudaMallocHost(&ctx->h_jout, n1 * sizeof(int)));
  ctx->max_lines = cap;
  return EKF_OK;
}

/* cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time libcuda dependency) */
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
int make_tensor_map(ekf_ctx* ctx, size_t p_rows, double* base, CUtensorMap* out, int pshape = -1) {
  void* fn = 0;
  cudaDriverEntryPointQueryResult q;
  CU(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
  if (!fn || q != cudaDriverEntryPointSuccess) { snprintf(ctx->err, sizeof ctx->err, "cuTensorMapEncodeTiled not available"); return EKF_ECUDA; }
  const cuuint64_t gdim[2] = {(cuuint64_t)ctx->g.ld, (cuuint64_t)p_rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)ctx->g.ld * sizeof(double)};
  int tr = 64, tc = 64;
  ekf_sweep_pbox(pshape >= 0 ? pshape : ctx->sweep_shape, &tr, &tc);
  const cuuint32_t box[2] = {(cuuint32_t)tc, (cuuint32_t)tr};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = ((EncodeTiledFn)fn)(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, base, gdim, gstride, box, estr,
                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { snprintf(ctx->err, sizeof ctx->err, "cuTensorMapEncodeTiled failed: %d", (int)r); return EKF_ECUDA; }
  return EKF_OK;
}

/* 2-D views of the pending lists: row = slot, inner dimension = 2*ld doubles (ld double2 entries) */
int make_band_map(ekf_ctx* ctx, double2* base, int box_entries, CUtensorMap* out) {
  void* fn = 0;
  cudaDriverEntryPointQueryResult q;
  CU(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
  if (!fn || q != cudaDriverEntryPointSuccess) { snprintf(ctx->err, sizeof ctx->err, "cuTensorMapEncodeTiled not available"); return EKF_ECUDA; }
  const cuuint64_t gdim[2] = {(cuuint64_t)2 * ctx->g.ld, (cuuint64_t)ctx->slots};
  const cuuint64_t gstride[1] = {(cuuint64_t)ctx->g.ld * sizeof(double2)};
  const cuuint32_t box[2] = {(cuuint32_t)(2 * box_entries), 8};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = ((EncodeTiledFn)fn)(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, base, gdim, gstride, box, estr,
                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { snprintf(ctx->err, sizeof ctx->err, "cuTensorMapEncodeTiled (band) failed: %d", (int)r); return EKF_ECUDA; }
  return EKF_OK;
}

int launch_sweep(ekf_ctx* ctx, int np_ub) {
  if (ctx->cfg.flags & EKF_FLAG_SWEEP_DIRECT) {
    CU(ekf_launch_sweep(ctx->g, ctx->b, 0, np_ub, ctx->L_ub, ctx->stream));
    ctx->launches++;
  } else {
    CU(ekf_launch_sweep_tma(ctx->g, ctx->b, &ctx->tmap2[ctx->rd], ctx->have_tmap8 ? &ctx->tmap8[ctx->rd] : 0, &ctx->tmapK[0], &ctx->tmapK[1], ctx->b.P, 0, 0, ctx->d_counters, ctx->sweep_shape, np_ub,
                            ctx->L_ub, ctx->num_sms, ctx->stream));
    const int per_pass = ekf_sweep_terms_per_pass(ctx->sweep_shape, np_ub);
    ctx->launches += (np_ub + per_pass - 1) / per_pass;
  }
  return EKF_OK;
}

int sweep_now(ekf_ctx* ctx, int np_ub) {
  if (np_ub <= 0) return EKF_OK;
  cudaEvent_t e0 = 0, e1 = 0;
  if (ctx->prof) {
    if (ctx->ev_used + 2 > ctx->ev.size()) {
      for (int i = 0; i < 64; ++i) { cudaEvent_t e; CU(cudaEventCreate(&e)); ctx->ev.push_back(e); }
    }
    e0 = ctx->ev[ctx->ev_used]; e1 = ctx->ev[ctx->ev_used + 1];
    CU(cudaEventRecord(e0, ctx->stream));
  }
  { int rc = launch_sweep(ctx, np_ub); if (rc) return rc; }
  if (ctx->prof) {
    CU(cudaEventRecord(e1, ctx->stream));
    ctx->ev_used += 2;
    ctx->ev_bytes.push_back((double)np_ub);   /* resolved to bytes at read time with the true n */
  }
  return EKF_OK;
}

/* exchange of the H-column slices in the row-sharded mode: every element of colA|colB has exactly one
 * non-zero contributor, so the sum is an exact gather */
int exchange_slices(ekf_ctx* ctx) {
  NcclApi* api = nccl_api();
  if (!api || !ctx->comm) { snprintf(ctx->err, sizeof ctx->err, "NCCL not available"); return EKF_ENCCL; }
  const int rc = api->AllReduce(ctx->b.colA, ctx->b.colA, 2 * (size_t)ctx->g.ld, kNcclFloat64, kNcclSum, ctx->comm, ctx->stream);
  if (rc != 0) {
    snprintf(ctx->err, sizeof ctx->err, "ncclAllReduce: %s", api->GetErrorString ? api->GetErrorString(rc) : "error");
    return EKF_ENCCL;
  }
  return EKF_OK;
}

/* gain + hot update for line `line` (j_sel: >= 0 explicit landmark, -1 association winner) */
int enqueue_update(ekf_ctx* ctx, const double* d_z, const double* d_R, int line, int j_sel) {
  if (ctx->pend_ub >= ctx->cfg.max_batch) {       /* fold what is pending before the list overflows */
    int rc = sweep_now(ctx, ctx->pend_ub);
    if (rc) return rc;
    CU(ekf_launch_flush_done(ctx->b, line, ctx->stream));
    ctx->launches++;
    ctx->pend_ub = 0;
  }
  if (ctx->g.world == 1) {
    CU(ekf_launch_gain(ctx->g, ctx->b, d_z, d_R, line, j_sel, 0, ctx->L_ub, ctx->cfg.max_batch, ctx->stream));
    ctx->launches++;
  } else {
    CU(ekf_launch_gain(ctx->g, ctx->b, d_z, d_R, line, j_sel, 1, ctx->L_ub, ctx->cfg.max_batch, ctx->stream));
    int rc = exchange_slices(ctx);
    if (rc) return rc;
    CU(ekf_launch_gain(ctx->g, ctx->b, d_z, d_R, line, j_sel, 2, ctx->L_ub, ctx->cfg.max_batch, ctx->stream));
    ctx->launches += 2;
  }
  CU(ekf_launch_apply(ctx->g, ctx->b, line, j_sel, ctx->L_ub, ctx->stream));
  ctx->launches++;
  ctx->pend_ub++;
  if (ctx->cfg.flags & EKF_FLAG_EAGER_SWEEP) {
    int rc = sweep_now(ctx, ctx->pend_ub);
    if (rc) return rc;
    CU(ekf_launch_flush_done(ctx->b, line + 1, ctx->stream));
    ctx->launches++;
    ctx->pend_ub = 0;
  }
  return EKF_OK;
}

int enqueue_end(ekf_ctx* ctx, const double* d_z, const double* d_R, int m) {
  int rc = sweep_now(ctx, ctx->pend_ub);
  if (rc) return rc;
  ctx->pend_ub = 0;
  CU(ekf_launch_end_scan(ctx->g, ctx->b, d_z, d_R, m, ctx->L_ub, 0, 0, ctx->stream));
  ctx->launches += (m > 0) ? 2 : 1;
  long long lub = (long long)ctx->L_ub + m;
  ctx->L_ub = (int)(lub > ctx->g.cap ? ctx->g.cap : lub);
  ctx->scan_open = 0;
  ctx->cursor = 0;
  return EKF_OK;
}

/* Waits for every sweep in flight and makes Pbuf[rd] the one complete, in-place-updatable covariance.
 * Everything except the overlapped ekf_scan path works on that view. */
int drain(ekf_ctx* ctx) {
  if (!ctx->overlap) return EKF_OK;
  { int rc = close_group(ctx); if (rc) return rc; }
  CU(cudaStreamSynchronize(ctx->wstream));
  if (ctx->pg_valid) { ctx->rd ^= 1; ctx->pg_valid = 0; }
  ctx->b.P = ctx->Pbuf[ctx->rd];
  ctx->evF_used[0] = ctx->evF_used[1] = 0;
  return EKF_OK;
}

int line_event(ekf_ctx* ctx) {
  if (!ctx->prof) return EKF_OK;
  if (ctx->lev_used + 1 > ctx->lev.size())
    for (int i = 0; i < 64; ++i) { cudaEvent_t e; CU(cudaEventCreate(&e)); ctx->lev.push_back(e); }
  CU(cudaEventRecord(ctx->lev[ctx->lev_used++], ctx->stream));
  return EKF_OK;
}

/* Hands the pending terms in slot half `par` (nterms: upper bound of their count, snapshot in d_view[par]) to the sweep
 * stream: the sweep reads the buffer the line stream has been appending to and writes the other one; then the next scan's
 * line loop reads that source buffer plus these terms, in the other half of the slot ring. */
int hand_off_sweep(ekf_ctx* ctx, int nterms, int L_ub, int line_sms) {
  const int par = ctx->par;
  const int slot0 = par * ctx->group;
  const int tgt = ctx->pg_valid ? (ctx->rd ^ 1) : ctx->rd;      /* source of this sweep */
  EkfBuffers bt = ctx->b;
  bt.P = ctx->Pbuf[tgt];
  CU(cudaEventRecord(ctx->evE, ctx->stream));
  CU(cudaStreamWaitEvent(ctx->wstream, ctx->evE, 0));
  cudaEvent_t e0 = 0, e1 = 0;
  if (ctx->prof) {
    if (ctx->ev_used + 2 > ctx->ev.size())
      for (int i = 0; i < 64; ++i) { cudaEvent_t e; CU(cudaEventCreate(&e)); ctx->ev.push_back(e); }
    e0 = ctx->ev[ctx->ev_used]; e1 = ctx->ev[ctx->ev_used + 1];
    CU(cudaEventRecord(e0, ctx->wstream));
  }
  CU(ekf_launch_sweep_tma(ctx->g, bt, &ctx->tmap2[tgt], ctx->have_tmap8 ? &ctx->tmap8[tgt] : 0, &ctx->tmapK[0], &ctx->tmapK[1], ctx->Pbuf[tgt ^ 1], slot0, &ctx->d_view[par], ctx->d_counters + 16,
                          ctx->sweep_shape, nterms, L_ub, ctx->num_sms - line_sms, ctx->wstream,
                          &ctx->tmap2[tgt ^ 1], ctx->have_tmap8 ? &ctx->tmap8[tgt ^ 1] : 0));
  { const int per_pass = ekf_sweep_terms_per_pass(ctx->sweep_shape, nterms); ctx->launches += (nterms + per_pass - 1) / per_pass; }
  if (ctx->prof) {
    CU(cudaEventRecord(e1, ctx->wstream));
    ctx->ev_used += 2;
    ctx->ev_bytes.push_back((double)nterms);
  }
  CU(cudaEventRecord(ctx->evF[par], ctx->wstream));
  ctx->evF_used[par] = 1;
  ctx->rd = tgt; ctx->pg_valid = 1; ctx->pg_slot0 = slot0;
  ctx->par ^= 1;
  ctx->b.P = ctx->Pbuf[ctx->rd];
  return EKF_OK;
}

/* launches the sweep of the open group, if any: after it nothing is owed but work already on the streams */
int close_group(ekf_ctx* ctx) {
  if (!ctx->grp_open) return EKF_OK;
  ctx->grp_open = 0;
  return hand_off_sweep(ctx, ctx->grp_terms, ctx->L_ub, ctx->grp_line_sms);
}

/* Overlapped form of one Robot::localize (single GPU, m <= group): the line stream runs predict, the
 * line-loop cluster kernel and the end-of-scan kernels against Pbuf[rd] plus the previous group's still
 * pending terms; the sweep of THIS scan's group is handed to the sweep stream when the group closes, where it
 * runs while the next group's line loops already execute.  Buffers: sweep(G) reads X and writes X^1; the next
 * group's line loops read X (complete once sweep(G-1) is done) plus G's pending terms. */
int enqueue_scan_overlapped(ekf_ctx* ctx, const double* d_u, const double* d_x_t0, int m, const double* d_z, const double* d_R) {
  /* Scans of more than chunk_above (32) lines go through the pipeline as CHUNKS of chunk_lines (16): a chunk's sweep (16 pending terms,
   * one tensor-core pass) runs while the next chunk's line loop executes, exactly as a scan's sweep runs under the next
   * scan's line loop.  A line then corrects its column reads against at most 2 x 16 pending terms instead of up to 128, and
   * the sweeps of a 64-line scan hide under its own line loop.  Prediction runs before the first chunk, the end-of-scan
   * kernels after the last; in between k_chunk_mark snapshots the finished chunk for its sweep and restarts the pending
   * list.  Same operations per element in the same order as one line loop + one sweep: identical bits. */
  const bool chunked = ctx->chunk_lines > 0 && m > ctx->chunk_above && ctx->g.world == 1;
  const int chunk = chunked ? ctx->chunk_lines : m;
  const int line_sms = line_sms_for(ctx->g.world, ctx->g.cap, m);
  /* Sweep groups (single GPU, unchunked scans): the scan joins the open group if its terms still fit the budget and its line
   * loop has the group's width; otherwise the open group is swept first and the scan starts a new one. */
  const bool groupable = ctx->grp_budget > 0 && !chunked && ctx->g.world == 1;
  const bool joins = groupable && ctx->grp_open && ctx->grp_terms + m <= ctx->grp_budget && line_sms == ctx->grp_line_sms;
  if (!joins) { int rc = close_group(ctx); if (rc) return rc; }
  const int grp_terms = joins ? ctx->grp_terms + m : m;
  /* the group stays open after this scan if one more scan of the same size would still fit */
  const bool stays_open = groupable && grp_terms + m <= ctx->grp_budget;
  /* the sweep still in flight was sized to leave last_line_sms SMs free: a wider line loop waits for it (only when the
   * number of lines per scan changes class) */
  if (line_sms > ctx->last_line_sms && ctx->pg_valid && ctx->evF_used[ctx->par ^ 1])
    CU(cudaStreamWaitEvent(ctx->stream, ctx->evF[ctx->par ^ 1], 0));
  ctx->last_line_sms = line_sms;
  use_tables(ctx, ctx->tabpar);
  ctx->tabpar ^= 1;
  long long lub = (long long)ctx->L_ub + m;
  const int L_after_ub = (int)(lub > ctx->g.cap ? ctx->g.cap : lub);
  { int rc = line_event(ctx); if (rc) return rc; }
  for (int line0 = 0; line0 < m; line0 += chunk) {
    const int line1 = line0 + chunk < m ? line0 + chunk : m;
    const bool first = line0 == 0, last = line1 == m;
    const int par = ctx->par;
    if (ctx->evF_used[par]) CU(cudaStreamWaitEvent(ctx->stream, ctx->evF[par], 0));   /* the sweep two back: slots free, X complete */
    const int slot0 = par * ctx->group;
    EkfBuffers b = ctx->b;
    b.P = ctx->Pbuf[ctx->rd];
    /* a scan that continues the group appends its terms after the group's earlier ones (their count: d_view[par].cnt) */
    const int* carry = joins ? &ctx->d_view[par].cnt : 0;
    const bool fuse = first && ekf_scan_lines_fuses_predict(ctx->peers_ok ? &ctx->peers : 0) && !ctx->no_fuse;
    if (first && !fuse) { CU(ekf_launch_predict(ctx->g, b, d_u, d_x_t0, m, ctx->L_ub, ctx->stream, carry)); ctx->launches++; }
    /* The line loop runs as line_sms cooperative CTAs on the SMs the in-flight sweep leaves free (its
     * persistent grid is num_sms - line_sms): no register / FP64-issue sharing with the sweep. */
    CU(ekf_launch_scan_lines(ctx->g, b, d_z, d_R, line0, line1, line_sms, 1, slot0, ctx->pg_slot0,
                             ctx->pg_valid ? &ctx->d_view[par ^ 1].cnt : 0, ctx->peers_ok ? &ctx->peers : 0, ctx->L_ub, ctx->stream,
                             fuse ? d_u : 0, fuse ? d_x_t0 : 0, m, fuse ? carry : 0));
    ctx->launches++;
    const int tgt = ctx->pg_valid ? (ctx->rd ^ 1) : ctx->rd;      /* source of the next sweep */
    EkfBuffers bt = ctx->b;
    bt.P = ctx->Pbuf[tgt];
    if (last) {
      /* After a map reset earlier in the group, the new landmarks reuse rows and columns that are live for the sweep still
       * in flight (it writes Pbuf[tgt] and reads Pbuf[rd] there): the end of this scan waits for that sweep. */
      if (joins && ctx->grp_may_reset && ctx->pg_valid && ctx->evF_used[par ^ 1])
        CU(cudaStreamWaitEvent(ctx->stream, ctx->evF[par ^ 1], 0));
      /* while the group stays open, the next scan reads Pbuf[rd] (not the sweep's source) and corrects against the previous
       * group's terms at every landmark, the new ones included */
      const bool keep = stays_open && tgt != ctx->rd;
      CU(ekf_launch_end_scan(ctx->g, bt, d_z, d_R, m, ctx->L_ub, slot0, &ctx->d_view[par], ctx->stream,
                             keep ? ctx->Pbuf[ctx->rd] : 0, ctx->pg_slot0, (stays_open && ctx->pg_valid) ? &ctx->d_view[par ^ 1].cnt : 0));
      ctx->launches += 2;
      int rc = line_event(ctx); if (rc) return rc;
    } else {
      CU(ekf_launch_chunk_mark(ctx->b, line1, &ctx->d_view[par], ctx->stream));
      ctx->launches++;
    }
    if (!groupable) { int rc = hand_off_sweep(ctx, line1 - line0, L_after_ub, line_sms); if (rc) return rc; }
  }
  if (groupable) {
    ctx->grp_may_reset = (joins && ctx->grp_may_reset) || (long long)ctx->L_ub + m > (long long)ctx->g.cap - ctx->g.headroom;
    ctx->grp_open = 1; ctx->grp_terms = grp_terms; ctx->grp_line_sms = line_sms;
  }
  ctx->L_ub = L_after_ub;
  ctx->b.P = ctx->Pbuf[ctx->rd];
  if (ctx->grp_open && !stays_open) return close_group(ctx);
  return EKF_OK;
}

/* the whole Robot::localize, enqueued without returning to the host */
int enqueue_scan(ekf_ctx* ctx, const double* d_u, const double* d_x_t0, int m, const double* d_z, const double* d_R) {
  if (ctx->overlap) {
    /* small maps: the sweep is a few microseconds, nothing to hide -- the in-place path with the 16-CTA
     * cluster line loop is faster there (measured crossover: a few thousand state entries) */
    const bool chunked = ctx->chunk_lines > 0 && m > ctx->chunk_above && ctx->g.world == 1;
    if (m >= 1 && (m <= ctx->group || chunked) && ctx->L_ub > 0 && 3 + 2 * ctx->L_ub >= kOverlapMinN &&
        (ctx->g.world == 1 || ctx->peers_ok))     /* a row-sharded filter overlaps only on the fused exchange */
      return enqueue_scan_overlapped(ctx, d_u, d_x_t0, m, d_z, d_R);
    int rc = drain(ctx);
    if (rc) return rc;
    use_tables(ctx, 0);
  }
  { int rc = line_event(ctx); if (rc) return rc; }
  /* fused path on a non-empty map: the prediction runs as the prologue of the line-loop launch (one launch less) */
  const bool fused_lines = ctx->L_ub > 0 && m > 0 && (ctx->g.world == 1 || ctx->peers_ok) && ctx->cfg.max_batch <= 64 &&
                           !(ctx->cfg.flags & (EKF_FLAG_EAGER_SWEEP | EKF_FLAG_PER_LINE_KERNELS));
  const bool fuse = fused_lines && ekf_scan_lines_fuses_predict(ctx->peers_ok ? &ctx->peers : 0) && !ctx->no_fuse;
  if (!fuse) {
    CU(ekf_launch_predict(ctx->g, ctx->b, d_u, d_x_t0, m, ctx->L_ub, ctx->stream));
    ctx->launches++;
  }
  ctx->pend_ub = 0;
  ctx->scan_open = 1;
  if (ctx->L_ub == 0) {
    CU(ekf_launch_queue_all(ctx->g, ctx->b, m, ctx->stream));
    if (m > 0) ctx->launches++;
  } else if ((ctx->g.world == 1 || ctx->peers_ok) && ctx->cfg.max_batch <= 64 &&
             !(ctx->cfg.flags & (EKF_FLAG_EAGER_SWEEP | EKF_FLAG_PER_LINE_KERNELS))) {
    /* fused: all lines in one cluster launch; split only where the pending list would overflow */
    int i0 = 0;
    while (i0 < m) {
      int cnt = ctx->cfg.max_batch - ctx->pend_ub;
      if (cnt > m - i0) cnt = m - i0;
      /* row-sharded: the same kernel, launched cooperatively (its CTAs spin on the peers' arrival flags, so they
       * must all be resident), exchanges the H-column slices over NVLink peer memory between its phases */
      CU(ekf_launch_scan_lines(ctx->g, ctx->b, d_z, d_R, i0, i0 + cnt, ctx->cluster, ctx->peers_ok ? 1 : 0, 0, 0, 0,
                               ctx->peers_ok ? &ctx->peers : 0, ctx->L_ub, ctx->stream,
                               (fuse && i0 == 0) ? d_u : 0, (fuse && i0 == 0) ? d_x_t0 : 0, m));
      ctx->launches++;
      ctx->pend_ub += cnt;
      i0 += cnt;
      if (i0 < m) {
        int rc = sweep_now(ctx, ctx->pend_ub);
        if (rc) return rc;
        CU(ekf_launch_flush_done(ctx->b, i0, ctx->stream));
        ctx->launches++;
        ctx->pend_ub = 0;
      }
    }
  } else {
    for (int i = 0; i < m; ++i) {
      CU(ekf_launch_associate(ctx->g, ctx->b, d_z, d_R, i, ctx->L_ub, ctx->stream));
      ctx->launches++;
      int rc = enqueue_update(ctx, d_z, d_R, i, -1);
      if (rc) return rc;
    }
  }
  { int rc = line_event(ctx); if (rc) return rc; }
  return enqueue_end(ctx, d_z, d_R, m);
}

int read_state(ekf_ctx* ctx) {
  CU(cudaMemcpyAsync(ctx->h_st, ctx->b.st, sizeof(EkfDevState), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (!ctx->scan_open) ctx->L_ub = ctx->h_st->L;
  ctx->snap_inflight = 0;                          /* the exact value supersedes any snapshot still on its way */
  return EKF_OK;
}

int sticky_to_status(int sticky) {
  if (sticky & EKF_STICKY_XCHG) return EKF_ENCCL;
  if (sticky & EKF_STICKY_CAPACITY) return EKF_ECAPACITY;
  if (sticky & EKF_STICKY_SINGULAR) return EKF_ESINGULAR;
  return EKF_OK;
}

/* Second covariance buffer, sweep stream and events of the overlapped pipeline (enqueue_scan_overlapped). */
int enable_overlap(ekf_ctx* ctx) {
  if (ctx->overlap) return EKF_OK;
  if (ctx->cfg.max_batch < 16 ||
      (ctx->cfg.flags & (EKF_FLAG_EAGER_SWEEP | EKF_FLAG_PER_LINE_KERNELS | EKF_FLAG_SWEEP_DIRECT | EKF_FLAG_NO_OVERLAP)))
    return EKF_OK;
  const size_t bytes = (size_t)ekf_local_tile_rows(ctx->g) * EKF_TILE * (size_t)ctx->g.ld * sizeof(double);
  if (cudaMalloc(&ctx->Pbuf[1], bytes) != cudaSuccess) {
    /* no room for the second covariance buffer (e.g. a 40k-landmark filter on too few GPUs): stay on the in-place,
     * non-overlapped path -- slower, same results */
    (void)cudaGetLastError();
    ctx->Pbuf[1] = 0;
    snprintf(ctx->err, sizeof ctx->err, "no memory for the second covariance buffer (%.1f GB): sweeps will not overlap", bytes / 1e9);
    return EKF_OK;
  }
  CU(cudaMemsetAsync(ctx->Pbuf[1], 0, bytes, ctx->stream));
  CU(cudaStreamCreateWithFlags(&ctx->wstream, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&ctx->evE, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&ctx->evF[0], cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&ctx->evF[1], cudaEventDisableTiming));
  { int rc = make_tensor_map(ctx, (size_t)ekf_local_tile_rows(ctx->g) * EKF_TILE, ctx->Pbuf[1], &ctx->tmap2[1]); if (rc) return rc; }
  if (ctx->have_tmap8) { int rc = make_tensor_map(ctx, (size_t)ekf_local_tile_rows(ctx->g) * EKF_TILE, ctx->Pbuf[1], &ctx->tmap8[1], 10); if (rc) return rc; }
  ekf_prefer_max_smem_carveout();
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->rd = 0; ctx->par = 0; ctx->pg_valid = 0;
  ctx->overlap = 1;
  /* L2 residency of the line loop's working set while sweeps stream the covariance through the cache (EKF_L2_PERSIST=0: off) */
  { const char* e = getenv("EKF_L2_PERSIST");
    const int mode = e ? atoi(e) : 0;
    if (mode >= 1) {
      int max_persist = 0, max_win = 0;
      cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, ctx->cfg.device);
      cudaDeviceGetAttribute(&max_win, cudaDevAttrMaxAccessPolicyWindowSize, ctx->cfg.device);
      size_t win = ctx->arena_bytes < (size_t)max_win ? ctx->arena_bytes : (size_t)max_win;
      size_t persist = win < (size_t)max_persist ? win : (size_t)max_persist;
      if (mode == 2) { win = (size_t)((char*)ctx->b.Kp - (char*)ctx->arena); persist = win; }        /* the small arrays only */
      if (mode >= 3) { persist = (size_t)mode << 20; if (persist > (size_t)max_persist) persist = max_persist; }   /* mode = MB set aside */
      if (win > 0 && persist > 0 && cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, persist) == cudaSuccess) {
        cudaStreamAttrValue av;
        memset(&av, 0, sizeof av);
        av.accessPolicyWindow.base_ptr = ctx->arena;
        av.accessPolicyWindow.num_bytes = win;
        av.accessPolicyWindow.hitRatio = (float)((double)persist / (double)win);
        av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        av.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
        if (cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &av) != cudaSuccess) (void)cudaGetLastError();
        if (getenv("EKF_VERBOSE")) fprintf(stderr, "libekfcuda: L2 window %.1f MB of arena %.1f MB, persisting %.1f MB (device max %.1f MB, window max %.1f MB)\n",
                                           win / 1e6, ctx->arena_bytes / 1e6, persist / 1e6, max_persist / 1e6, max_win / 1e6);
      } else (void)cudaGetLastError();
    } }
  return EKF_OK;
}

int create_common(ekf_ctx** out, const ekf_config* cfg, int rank, int world, const unsigned char* uid) {
  if (!out || !cfg || cfg->capacity_lines < 1 || cfg->reset_headroom < 0 || world < 1 || rank < 0 || rank >= world)
    return EKF_EINVAL;
  ekf_ctx* ctx = new ekf_ctx();
  memset(&ctx->b, 0, sizeof ctx->b);
  ctx->cfg = *cfg;
  if (ctx->cfg.max_batch <= 0) ctx->cfg.max_batch = 64;
  ctx->err[0] = 0;
  ctx->stream = 0; ctx->max_lines = 0; ctx->d_in = 0; ctx->h_in = 0; ctx->h_jout = 0; ctx->h_st = 0;
  ctx->L_ub = 0; ctx->pend_ub = 0; ctx->scan_open = 0; ctx->cursor = 0;
  ctx->prof = 0; ctx->ev_used = 0; ctx->lev_used = 0; ctx->launches = 0; ctx->comm = 0; ctx->t0 = 0; ctx->t1 = 0;
  ctx->d_stage = 0; ctx->stage_elems = 0; ctx->d_partials = 0; ctx->d_out3 = 0; ctx->d_keep = 0;
  ctx->overlap = 0; ctx->wstream = 0; ctx->Pbuf[0] = ctx->Pbuf[1] = 0; ctx->rd = 0; ctx->par = 0; ctx->group = 8; ctx->tabpar = 0;
  { const char* e = getenv("EKF_CHUNK"); ctx->chunk_lines = e ? atoi(e) : 16; if (ctx->chunk_lines < 0) ctx->chunk_lines = 0; }
  { const char* e = getenv("EKF_FUSE_PREDICT"); ctx->no_fuse = (e && atoi(e) == 0) ? 1 : 0; }
  { const char* e = getenv("EKF_CHUNK_ABOVE"); ctx->chunk_above = e ? atoi(e) : 32; if (ctx->chunk_above < 1) ctx->chunk_above = 1; }
  ctx->pg_valid = 0; ctx->pg_slot0 = 0; ctx->d_view = 0;
  ctx->grp_open = 0; ctx->grp_terms = 0; ctx->grp_line_sms = 0; ctx->grp_may_reset = 0; ctx->d_counters = 0; ctx->evE = 0; ctx->evF[0] = ctx->evF[1] = 0;
  ctx->evF_used[0] = ctx->evF_used[1] = 0; memset(ctx->tab, 0, sizeof ctx->tab);
  ctx->last_line_sms = 64; ctx->arena = 0; ctx->arena_bytes = 0; ctx->h_snap = 0; ctx->ev_snap = 0; ctx->snap_inflight = 0; ctx->snap_added = 0; ctx->xchg = 0; ctx->poisoned = 0; ctx->peers_ok = 0; ctx->peers_mapped = 0; memset(ctx->peer_map, 0, sizeof ctx->peer_map); memset(&ctx->peers, 0, sizeof ctx->peers);
  *out = ctx;                                  /* so the caller can read ekf_last_error on failure */
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    snprintf(ctx->err, sizeof ctx->err, "no CUDA device: libekfcuda has no CPU fallback");
    return EKF_ECUDA;
  }
  CU(cudaSetDevice(cfg->device));
  EkfGeom& g = ctx->g;
  g.cap = cfg->capacity_lines;
  g.n = 3 + 2 * g.cap;
  g.ld = ((g.n + EKF_LD_ALIGN - 1) / EKF_LD_ALIGN) * EKF_LD_ALIGN;
  g.rank = rank; g.world = world;
  g.gate = cfg->gate; g.enc_noise = cfg->encoder_noise; g.headroom = cfg->reset_headroom;
  g.gate_d2max = ekf_gate_d2max(cfg->gate);
  CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  const size_t ld = g.ld;
  const size_t p_rows = (size_t)ekf_local_tile_rows(g) * EKF_TILE;
  CU(cudaMalloc(&ctx->b.st, sizeof(EkfDevState)));
  CU(cudaMalloc(&ctx->b.P, p_rows * ld * sizeof(double)));
  ctx->Pbuf[0] = ctx->b.P; ctx->Pbuf[1] = 0;
  ctx->overlap = 0;
  /* lines per overlapped scan: the pending-slot ring holds two scans' terms ([2][group] slots) and one out-of-place
   * sweep pass folds at most 32 */
  /* from max_batch = 64 on (the default) an overlapped scan may hold up to 64 lines: its sweep is then two chained passes */
  ctx->group = ctx->cfg.max_batch >= 64 ? 64 : (ctx->cfg.max_batch / 2 < 32 ? ctx->cfg.max_batch / 2 : 32);
  ctx->slots = ctx->cfg.max_batch > 2 * ctx->group ? ctx->cfg.max_batch : 2 * ctx->group;
  CU(cudaMalloc(&ctx->d_counters, 32 * sizeof(unsigned long long)));
  CU(cudaMalloc(&ctx->d_view, 2 * sizeof(EkfScanView)));
  CU(cudaMemsetAsync(ctx->d_view, 0, 2 * sizeof(EkfScanView), ctx->stream));
  {
    /* Everything the line loop reads and writes -- the hot state, the gate records, the pending lists -- lives in ONE
     * allocation, so that one L2 access-policy window can cover it (enable_overlap): beside a sweep that streams 6.4 GB
     * through the L2 per pass, these few MB are what every dependent round trip of a line waits for. */
    const size_t al = 256;
    auto up = [&](size_t x) { return (x + al - 1) / al * al; };
    const size_t o_y = 0, o_top = o_y + up(ld * sizeof(double)), o_diag = o_top + up(3 * ld * sizeof(double)),
                 o_gates = o_diag + up(4 * (size_t)g.cap * sizeof(double)), o_matched = o_gates + up(24 * (size_t)g.cap * sizeof(double)),
                 o_col = o_matched + up((size_t)g.cap * sizeof(int)), o_kp = o_col + up(2 * ld * sizeof(double)),
                 o_ksp = o_kp + up((size_t)ctx->slots * ld * sizeof(double2)), total = o_ksp + up((size_t)ctx->slots * ld * sizeof(double2));
    CU(cudaMalloc(&ctx->arena, total));
    ctx->arena_bytes = total;
    char* a = (char*)ctx->arena;
    ctx->b.y = (double*)(a + o_y); ctx->b.top = (double*)(a + o_top); ctx->b.diag = (double*)(a + o_diag);
    ctx->b.gates = (double*)(a + o_gates);                                  /* GATE_REC doubles per landmark */
    ctx->b.matched = (int*)(a + o_matched);
    ctx->b.colA = (double*)(a + o_col); ctx->b.colB = ctx->b.colA + ld;
    ctx->b.Kp = (double2*)(a + o_kp); ctx->b.KSp = (double2*)(a + o_ksp);
  }
  CU(cudaMallocHost(&ctx->h_st, sizeof(EkfDevState)));
  CU(cudaMallocHost(&ctx->h_snap, sizeof(EkfDevState)));
  CU(cudaEventCreateWithFlags(&ctx->ev_snap, cudaEventDisableTiming));
  CU(cudaDeviceGetAttribute(&ctx->num_sms, cudaDevAttrMultiProcessorCount, cfg->device));
  { const char* e = getenv("EKF_SWEEP_SHAPE"); ctx->sweep_shape = e ? atoi(e) : 0; if (ctx->sweep_shape < 0 || (ctx->sweep_shape > 5 && ctx->sweep_shape != 8 && ctx->sweep_shape != 9 && ctx->sweep_shape != 10 && ctx->sweep_shape != 11) || ctx->sweep_shape == 3) ctx->sweep_shape = 0; }
  { const int cap = 2 * ekf_sweep_terms_per_pass(ctx->sweep_shape, 64); if (ctx->group > cap) ctx->group = cap; if (ctx->group < 1) ctx->group = 1; }
  if (ctx->chunk_lines > ctx->group) ctx->chunk_lines = ctx->group;          /* a chunk's terms live in one half of the slot ring */
  /* Terms per sweep group: 16, the largest pass that is still HBM-bound at 10k landmarks (DESIGN section 4.1: 0.504 ms
   * against 0.491 for 8 terms).  A group's terms live in one half of the slot ring, and a line corrects against the previous
   * group's terms plus its own group's: both fit the ring half (group) and FL_MAXP (128 >= 2 x group). */
  { const char* e = getenv("EKF_SWEEP_GROUP"); ctx->grp_budget = e ? atoi(e) : 16; }
  if (ctx->grp_budget < 0) ctx->grp_budget = 0;
  if (ctx->grp_budget > ctx->group) ctx->grp_budget = ctx->group;
  { int rc = make_tensor_map(ctx, p_rows, ctx->Pbuf[0], &ctx->tmap2[0]); if (rc) return rc; }
  ctx->have_tmap8 = (ctx->sweep_shape == 0 || ctx->sweep_shape == 10);
  if (ctx->have_tmap8) { int rc = make_tensor_map(ctx, p_rows, ctx->Pbuf[0], &ctx->tmap8[0], 10); if (rc) return rc; }
  { int tr = 64, tc = 64; ekf_sweep_shape(ctx->sweep_shape, &tr, &tc);
    int rc = make_band_map(ctx, ctx->b.Kp, tc, &ctx->tmapK[0]); if (rc) return rc;
    rc = make_band_map(ctx, ctx->b.KSp, tr, &ctx->tmapK[1]); if (rc) return rc; }
  ctx->cluster = ekf_pick_cluster();
  /* a row-sharded filter overlaps only once its peers are connected (ekf_shard_connect) */
  if (world == 1) { int rc = enable_overlap(ctx); if (rc) return rc; }
  CU(cudaMalloc(&ctx->d_partials, 3 * (size_t)g.n * sizeof(double)));
  CU(cudaMalloc(&ctx->d_out3, 3 * sizeof(double)));
  CU(cudaMemsetAsync(ctx->b.st, 0, sizeof(EkfDevState), ctx->stream));
  CU(cudaMemsetAsync(ctx->b.y, 0, ld * sizeof(double), ctx->stream));
  CU(cudaMemsetAsync(ctx->b.top, 0, 3 * ld * sizeof(double), ctx->stream));
  CU(cudaMemsetAsync(ctx->b.diag, 0, 4 * (size_t)g.cap * sizeof(double), ctx->stream));
  CU(cudaMemsetAsync(ctx->b.P, 0, p_rows * ld * sizeof(double), ctx->stream));
  CU(cudaMemsetAsync(ctx->b.matched, 0, (size_t)g.cap * sizeof(int), ctx->stream));
  CU(cudaMemsetAsync(ctx->b.Kp, 0, (size_t)ctx->slots * ld * sizeof(double2), ctx->stream));
  CU(cudaMemsetAsync(ctx->b.KSp, 0, (size_t)ctx->slots * ld * sizeof(double2), ctx->stream));
  CU(cudaMemsetAsync(ctx->b.colA, 0, 2 * ld * sizeof(double), ctx->stream));
  int rc = ensure_lines(ctx, 64);
  if (rc) return rc;
  CU(ekf_launch_init(g, ctx->b, ctx->stream));
  if (world > 1) {
    if (world <= 8) {     /* exchange buffer of the in-kernel NVLink path (mapped by the peers through CUDA IPC) */
      const size_t xb = (4 * ld + 16) * sizeof(double);
      CU(cudaMalloc(&ctx->xchg, xb));
      CU(cudaMemsetAsync(ctx->xchg, 0, xb, ctx->stream));
    }
    NcclApi* api = nccl_api();
    if (!api || !uid) { snprintf(ctx->err, sizeof ctx->err, "libnccl.so.2 could not be loaded"); return EKF_ENCCL; }
    ncclUniqueId id;
    memcpy(id.internal, uid, 128);
    const int nrc = api->CommInitRank(&ctx->comm, world, id, rank);
    if (nrc != 0) {
      snprintf(ctx->err, sizeof ctx->err, "ncclCommInitRank: %s", api->GetErrorString ? api->GetErrorString(nrc) : "error");
      return EKF_ENCCL;
    }
  }
  CU(cudaStreamSynchronize(ctx->stream));
  return EKF_OK;
}

int ensure_stage(ekf_ctx* ctx, size_t elems) {
  if (elems <= ctx->stage_elems) return EKF_OK;
  if (ctx->d_stage) cudaFree(ctx->d_stage);
  ctx->d_stage = 0; ctx->stage_elems = 0;
  CU(cudaMalloc(&ctx->d_stage, elems * sizeof(double)));
  ctx->stage_elems = elems;
  return EKF_OK;
}

/* rows [0,nr) x cols [0,nc) of the symmetrised covariance into host memory with row stride ldp */
int download_rect(ekf_ctx* ctx, int r0, int c0, int nr, int nc, double* P, size_t ldp) {
  if (nr <= 0 || nc <= 0) return EKF_OK;
  size_t rows_per = kStageElems / (size_t)nc;
  if (rows_per < 1) rows_per = 1;
  if (rows_per > (size_t)nr) rows_per = nr;
  int rc = ensure_stage(ctx, rows_per * (size_t)nc);
  if (rc) return rc;
  for (int r = 0; r < nr; r += (int)rows_per) {
    const int cnt = (nr - r < (int)rows_per) ? nr - r : (int)rows_per;
    CU(ekf_launch_assemble(ctx->g, ctx->b, r0 + r, cnt, c0, nc, ctx->d_stage, nc, ctx->stream));
    CU(cudaMemcpy2DAsync(P + (size_t)r * ldp, ldp * sizeof(double), ctx->d_stage, (size_t)nc * sizeof(double),
                         (size_t)nc * sizeof(double), cnt, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  return EKF_OK;
}

}  // namespace

extern "C" {

const char* ekf_version(void) { return "libekfcuda 0.1 (sm_100a)"; }

int ekf_default_config(ekf_config* cfg) {
  if (!cfg) return EKF_EINVAL;
  cfg->capacity_lines = 100;      /* Robot.h:13 */
  cfg->gate = 0.4;                /* Robot.h:15 */
  cfg->encoder_noise = 0.024;     /* Robot.h:17 */
  cfg->reset_headroom = 10;       /* Robot.cpp:893 */
  cfg->device = 0;
  cfg->max_batch = 64;
  cfg->flags = 0;
  return EKF_OK;
}

int ekf_create(ekf_ctx** out, const ekf_config* cfg) { return create_common(out, cfg, 0, 1, 0); }

int ekf_nccl_unique_id(unsigned char id[128]) {
  NcclApi* api = nccl_api();
  if (!api || !id) return EKF_ENCCL;
  ncclUniqueId u;
  if (api->GetUniqueId(&u) != 0) return EKF_ENCCL;
  memcpy(id, u.internal, 128);
  return EKF_OK;
}

int ekf_create_sharded(ekf_ctx** out, const ekf_config* cfg, int rank, int world, const unsigned char uid[128]) {
  return create_common(out, cfg, rank, world, uid);
}

int ekf_shard_ipc_handle(ekf_ctx* ctx, unsigned char handle[64]) {
  if (!ctx || !handle) return EKF_EINVAL;
  if (!ctx->xchg) { snprintf(ctx->err, sizeof ctx->err, "not a row-sharded filter (or world > 8)"); return EKF_ESTATE; }
  CU(cudaSetDevice(ctx->cfg.device));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, ctx->xchg));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
  memcpy(handle, &h, 64);
  return EKF_OK;
}

int ekf_shard_connect(ekf_ctx* ctx, const unsigned char* handles) {
  if (!ctx || !handles) return EKF_EINVAL;
  if (!ctx->xchg) { snprintf(ctx->err, sizeof ctx->err, "not a row-sharded filter (or world > 8)"); return EKF_ESTATE; }
  if (ctx->scan_open) return EKF_ESTATE;
  if (ctx->peers_mapped) return EKF_OK;
  CU(cudaSetDevice(ctx->cfg.device));
  const int world = ctx->g.world, rank = ctx->g.rank;
  memset(&ctx->peers, 0, sizeof ctx->peers);
  ctx->peers.world = world; ctx->peers.rank = rank;
  for (int p = 0; p < world; ++p) {
    if (p == rank) { ctx->peers.xchg[p] = ctx->xchg; continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + 64 * (size_t)p, 64);
    void* ptr = 0;
    const cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      snprintf(ctx->err, sizeof ctx->err, "cudaIpcOpenMemHandle(rank %d): %s -- staying on the NCCL exchange", p, cudaGetErrorString(e));
      for (int q = 0; q < p; ++q) if (ctx->peer_map[q]) { cudaIpcCloseMemHandle(ctx->peer_map[q]); ctx->peer_map[q] = 0; }
      return EKF_ECUDA;
    }
    ctx->peer_map[p] = ptr;
    ctx->peers.xchg[p] = (double*)ptr;
  }
  ctx->peers_mapped = 1;
  return EKF_OK;
}

int ekf_shard_use_fused(ekf_ctx* ctx, int on) {
  if (!ctx) return EKF_EINVAL;
  if (ctx->scan_open) return EKF_ESTATE;
  if (on && !ctx->peers_mapped) { snprintf(ctx->err, sizeof ctx->err, "ekf_shard_use_fused before a successful ekf_shard_connect"); return EKF_ESTATE; }
  CU(cudaSetDevice(ctx->cfg.device));
  { int rc = drain(ctx); if (rc) return rc; }
  ctx->peers_ok = on ? 1 : 0;
  return on ? enable_overlap(ctx) : EKF_OK;
}

int ekf_destroy(ekf_ctx* ctx) {
  if (!ctx) return EKF_EINVAL;
  cudaSetDevice(ctx->cfg.device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->wstream) cudaStreamSynchronize(ctx->wstream);
  if (ctx->comm) { NcclApi* api = nccl_api(); if (api) api->CommDestroy(ctx->comm); }
  for (int p = 0; p < 8; ++p) if (ctx->peer_map[p]) cudaIpcCloseMemHandle(ctx->peer_map[p]);
  cudaFree(ctx->xchg);
  free_line_tables(ctx);
  cudaFree(ctx->b.st); cudaFree(ctx->arena); cudaFree(ctx->Pbuf[0]); cudaFree(ctx->Pbuf[1]);
  cudaFree(ctx->d_view); cudaFree(ctx->d_counters);
  if (ctx->evE) cudaEventDestroy(ctx->evE);
  if (ctx->evF[0]) cudaEventDestroy(ctx->evF[0]);
  if (ctx->evF[1]) cudaEventDestroy(ctx->evF[1]);
  if (ctx->wstream) cudaStreamDestroy(ctx->wstream);
  cudaFree(ctx->d_stage); cudaFree(ctx->d_partials); cudaFree(ctx->d_out3); cudaFree(ctx->d_keep);
  cudaFreeHost(ctx->h_st); cudaFreeHost(ctx->h_snap);
  if (ctx->ev_snap) cudaEventDestroy(ctx->ev_snap);
  for (size_t i = 0; i < ctx->ev.size(); ++i) cudaEventDestroy(ctx->ev[i]);
  for (size_t i = 0; i < ctx->lev.size(); ++i) cudaEventDestroy(ctx->lev[i]);
  if (ctx->t0) cudaEventDestroy(ctx->t0);
  if (ctx->t1) cudaEventDestroy(ctx->t1);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return EKF_OK;
}

const char* ekf_last_error(const ekf_ctx* ctx) { return ctx ? ctx->err : "null ctx"; }

/* ------------------------------------------ fused path ------------------------------------------- */
int ekf_scan(ekf_ctx* ctx, const double x_t0[3], const double u[3], int m, const double* z, const double* R,
             int* j_out, double pose[3]) {
  if (!ctx || !u || m < 0 || (m > 0 && (!z || !R))) return EKF_EINVAL;
  if (ctx->scan_open) { snprintf(ctx->err, sizeof ctx->err, "ekf_scan inside an open step-wise scan"); return EKF_ESTATE; }
  NOT_POISONED(ctx);
  CU(cudaSetDevice(ctx->cfg.device));
  int rc = ensure_lines(ctx, m);
  if (rc) return rc;
  double* h = ctx->h_in;
  memcpy(h, u, 3 * sizeof(double));
  if (x_t0) memcpy(h + 3, x_t0, 3 * sizeof(double));
  const size_t ml = ctx->max_lines;
  if (m > 0) { memcpy(h + 6, z, 2 * (size_t)m * sizeof(double)); memcpy(h + 6 + 2 * ml, R, 4 * (size_t)m * sizeof(double)); }
  /* H2D from pinned memory: [u|x|z] and [R] -- as ONE copy spanning the unused z slots in between while that stays small
   * (one driver call less on the latency path of small maps), else as two */
  const size_t span = 6 + 2 * ml + 4 * (size_t)m;
  if (m > 0 && span * sizeof(double) <= 8192) {
    CU(cudaMemcpyAsync(ctx->d_in, h, span * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  } else {
    CU(cudaMemcpyAsync(ctx->d_in, h, (6 + 2 * (size_t)m) * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    if (m > 0) CU(cudaMemcpyAsync(in_R(ctx), h + 6 + 2 * ml, 4 * (size_t)m * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  }
  rc = enqueue_scan(ctx, in_u(ctx), x_t0 ? in_x(ctx) : 0, m, in_z(ctx), in_R(ctx));
  if (rc) return rc;
  if (m > 0 && j_out) CU(cudaMemcpyAsync(ctx->h_jout, ctx->b.jout, (size_t)m * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  rc = read_state(ctx);
  if (rc) return rc;
  if (m > 0 && j_out) memcpy(j_out, ctx->h_jout, (size_t)m * sizeof(int));
  if (pose) memcpy(pose, ctx->h_st->pose, 3 * sizeof(double));
  const int sticky = ctx->h_st->sticky;
  if (sticky) {
    CU(cudaMemsetAsync(&ctx->b.st->sticky, 0, sizeof(int), ctx->stream));
    snprintf(ctx->err, sizeof ctx->err, "scan finished with sticky status 0x%x", sticky);
    if (sticky & EKF_STICKY_XCHG) ctx->poisoned = 1;
  }
  return sticky_to_status(sticky);
}

int ekf_scan_device(ekf_ctx* ctx, const double* d_u, int m, const double* d_z, const double* d_R, int* d_j_out) {
  if (!ctx || !d_u || m < 0 || (m > 0 && (!d_z || !d_R))) return EKF_EINVAL;
  if (ctx->scan_open) return EKF_ESTATE;
  NOT_POISONED(ctx);
  CU(cudaSetDevice(ctx->cfg.device));
  int rc = ensure_lines(ctx, m);
  if (rc) return rc;
  if (ctx->snap_inflight && cudaEventQuery(ctx->ev_snap) == cudaSuccess) {
    const long long lub = (long long)ctx->h_snap->L + ctx->snap_added;
    if (lub < ctx->L_ub) ctx->L_ub = (int)lub;
    ctx->snap_inflight = 0;
  } else if (ctx->snap_inflight) (void)cudaGetLastError();            /* cudaErrorNotReady is not an error */
  rc = enqueue_scan(ctx, d_u, 0, m, d_z, d_R);
  if (rc) return rc;
  if (ctx->snap_inflight) ctx->snap_added += m;
  else {
    CU(cudaMemcpyAsync(ctx->h_snap, ctx->b.st, sizeof(EkfDevState), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaEventRecord(ctx->ev_snap, ctx->stream));
    ctx->snap_inflight = 1; ctx->snap_added = 0;
  }
  if (d_j_out && m > 0)
    CU(cudaMemcpyAsync(d_j_out, ctx->b.jout, (size_t)m * sizeof(int), cudaMemcpyDeviceToDevice, ctx->stream));
  return EKF_OK;
}

int ekf_sync(ekf_ctx* ctx) {
  if (!ctx) return EKF_EINVAL;
  CU(cudaSetDevice(ctx->cfg.device));
  { int rc = close_group(ctx); if (rc) return rc; }   /* returns with no work owed: the open sweep group is swept too */
  CU(cudaStreamSynchronize(ctx->stream));
  if (ctx->wstream) CU(cudaStreamSynchronize(ctx->wstream));
  return EKF_OK;
}

/* ---------------------------------------- step-wise path ----------------------------------------- */
int ekf_predict(ekf_ctx* ctx, const double x_t0[3], const double u[3], double x_pre[3]) {
  if (!ctx || !u) return EKF_EINVAL;
  if (ctx->scan_open) { snprintf(ctx->err, sizeof ctx->err, "ekf_predict: previous scan not ended"); return EKF_ESTATE; }
  NOT_POISONED(ctx);
  CU(cudaSetDevice(ctx->cfg.device));
  { int rc = drain(ctx); if (rc) return rc; }
  { int rc = ensure_lines(ctx, 1); if (rc) return rc; }     /* re-creates the line tables after a failed growth */
  use_tables(ctx, 0);
  double* h = ctx->h_in;
  memcpy(h, u, 3 * sizeof(double));
  if (x_t0) memcpy(h + 3, x_t0, 3 * sizeof(double));
  CU(cudaMemcpyAsync(ctx->d_in, h, 6 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CU(ekf_launch_predict(ctx->g, ctx->b, in_u(ctx), x_t0 ? in_x(ctx) : 0, ctx->max_lines, ctx->L_ub, ctx->stream));
  ctx->launches++;
  ctx->pend_ub = 0; ctx->scan_open = 1; ctx->cursor = 0;
  int rc = read_state(ctx);
  if (rc) return rc;
  if (x_pre) memcpy(x_pre, ctx->h_st->x_pre, 3 * sizeof(double));
  return EKF_OK;
}

namespace {
int stage_line(ekf_ctx* ctx, const double z[2], const double R[4]) {
  if (ctx->cursor >= ctx->max_lines) {
    snprintf(ctx->err, sizeof ctx->err, "more than %d lines in a step-wise scan (limit of the step-wise ABI, see ekf.h; ekf_scan has none)", ctx->max_lines);
    return EKF_EINVAL;
  }
  const int i = ctx->cursor;
  /* pinned slots mirror the device layout, so an earlier line's copy is never overwritten in flight */
  double* hz = ctx->h_in + 6 + 2 * (size_t)i;
  double* hR = ctx->h_in + 6 + 2 * (size_t)ctx->max_lines + 4 * (size_t)i;
  hz[0] = z[0]; hz[1] = z[1]; hR[0] = R[0]; hR[1] = R[1]; hR[2] = R[2]; hR[3] = R[3];
  CU(cudaMemcpyAsync(in_z(ctx) + 2 * (size_t)i, hz, 2 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(in_R(ctx) + 4 * (size_t)i, hR, 4 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  return EKF_OK;
}
}  // namespace

int ekf_associate(ekf_ctx* ctx, const double z[2], const double R[4], int* j_out, double innov[2]) {
  if (!ctx || !z || !R || !j_out) return EKF_EINVAL;
  if (!ctx->scan_open) { snprintf(ctx->err, sizeof ctx->err, "ekf_associate before ekf_predict"); return EKF_ESTATE; }
  NOT_POISONED(ctx);
  CU(cudaSetDevice(ctx->cfg.device));
  int rc = stage_line(ctx, z, R);
  if (rc) return rc;
  const int i = ctx->cursor;
  const int none = EKF_NO_MATCH;
  ctx->h_jout[0] = none;
  CU(cudaMemcpyAsync(ctx->b.jbest + i, ctx->h_jout, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(ctx->b.jsing + i, ctx->h_jout, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  CU(ekf_launch_associate(ctx->g, ctx->b, in_z(ctx), in_R(ctx), i, ctx->L_ub, ctx->stream));
  if (ctx->L_ub > 0) {
    CU(ekf_launch_gain(ctx->g, ctx->b, in_z(ctx), in_R(ctx), i, -1, 3, 1, ctx->cfg.max_batch, ctx->stream));
    ctx->launches += 2;
  }
  CU(cudaMemcpyAsync(ctx->h_jout, ctx->b.jbest + i, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  rc = read_state(ctx);
  if (rc) return rc;
  const int j = ctx->h_jout[0];
  *j_out = (j == EKF_NO_MATCH) ? -1 : j;
  if (innov) { innov[0] = (j == EKF_NO_MATCH) ? 0.0 : ctx->h_st->v[0]; innov[1] = (j == EKF_NO_MATCH) ? 0.0 : ctx->h_st->v[1]; }
  return EKF_OK;
}

int ekf_update(ekf_ctx* ctx, int j, const double z[2], const double R[4], double x_post[3]) {
  if (!ctx || !z || !R || j < 0) return EKF_EINVAL;
  if (!ctx->scan_open) { snprintf(ctx->err, sizeof ctx->err, "ekf_update before ekf_predict"); return EKF_ESTATE; }
  NOT_POISONED(ctx);
  CU(cudaSetDevice(ctx->cfg.device));
  int rc = read_state(ctx);
  if (rc) return rc;
  if (j >= ctx->h_st->L) { snprintf(ctx->err, sizeof ctx->err, "ekf_update: landmark %d >= %d", j, ctx->h_st->L); return EKF_EINVAL; }
  rc = stage_line(ctx, z, R);
  if (rc) return rc;
  rc = enqueue_update(ctx, in_z(ctx), in_R(ctx), ctx->cursor, j);
  if (rc) return rc;
  ctx->cursor++;
  if (x_post) {
    rc = read_state(ctx);
    if (rc) return rc;
    memcpy(x_post, ctx->h_st->pose, 3 * sizeof(double));
  }
  return EKF_OK;
}

int ekf_add_line(ekf_ctx* ctx, const double z[2], const double R[4]) {
  if (!ctx || !z || !R) return EKF_EINVAL;
  if (!ctx->scan_open) { snprintf(ctx->err, sizeof ctx->err, "ekf_add_line before ekf_predict"); return EKF_ESTATE; }
  CU(cudaSetDevice(ctx->cfg.device));
  int rc = stage_line(ctx, z, R);
  if (rc) return rc;
  CU(ekf_launch_apply(ctx->g, ctx->b, ctx->cursor, -2, 0, ctx->stream));
  ctx->launches++;
  ctx->cursor++;
  return EKF_OK;
}

int ekf_end_scan(ekf_ctx* ctx, int n_lines, double pose[3]) {
  if (!ctx) return EKF_EINVAL;
  if (!ctx->scan_open) { snprintf(ctx->err, sizeof ctx->err, "ekf_end_scan before ekf_predict"); return EKF_ESTATE; }
  if (n_lines != ctx->cursor) {
    snprintf(ctx->err, sizeof ctx->err, "ekf_end_scan: n_lines=%d but %d lines were updated/queued", n_lines, ctx->cursor);
    return EKF_EINVAL;
  }
  CU(cudaSetDevice(ctx->cfg.device));
  int rc = enqueue_end(ctx, in_z(ctx), in_R(ctx), n_lines);
  if (rc) return rc;
  rc = read_state(ctx);
  if (rc) return rc;
  if (pose) memcpy(pose, ctx->h_st->pose, 3 * sizeof(double));
  const int sticky = ctx->h_st->sticky;
  if (sticky) CU(cudaMemsetAsync(&ctx->b.st->sticky, 0, sizeof(int), ctx->stream));
  if (sticky & EKF_STICKY_XCHG) ctx->poisoned = 1;
  return sticky_to_status(sticky);
}

/* ------------------------------------------ state access ----------------------------------------- */
int ekf_get_state(ekf_ctx* ctx, double pose[3], int* n_lines, int* sticky_status) {
  if (!ctx) return EKF_EINVAL;
  CU(cudaSetDevice(ctx->cfg.device));
  int rc = read_state(ctx);
  if (rc) return rc;
  if (pose) memcpy(pose, ctx->h_st->pose, 3 * sizeof(double));
  if (n_lines) *n_lines = ctx->h_st->L;
  if (sticky_status) {
    *sticky_status = sticky_to_status(ctx->h_st->sticky);
    if (ctx->h_st->sticky & EKF_STICKY_XCHG) ctx->poisoned = 1;
    if (ctx->h_st->sticky) CU(cudaMemsetAsync(&ctx->b.st->sticky, 0, sizeof(int), ctx->stream));
  }
  return EKF_OK;
}

int ekf_get_robot_cov(ekf_ctx* ctx, double Prr[9]) {
  if (!ctx || !Prr) return EKF_EINVAL;
  CU(cudaSetDevice(ctx->cfg.device));
  double t[9];
  CU(cudaMemcpy2DAsync(t, 3 * sizeof(double), ctx->b.top, (size_t)ctx->g.ld * sizeof(double), 3 * sizeof(double), 3,
                       cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < 3; ++i)
    for (int k = 0; k < 3; ++k) Prr[3 * i + k] = (i <= k) ? t[3 * i + k] : t[3 * k + i];
  return EKF_OK;
}

int ekf_get_ellipse(ekf_ctx* ctx, float axii[2], float* angle, int* ok) {
  if (!ctx || !axii || !angle) return EKF_EINVAL;
  double Prr[9];
  int rc = ekf_get_robot_cov(ctx, Prr);
  if (rc) return rc;
  /* Robot.cpp:75-113 on the 2x2 block: closed-form eigen-decomposition (symmetric input) */
  const double a = Prr[0], b = Prr[1], c = Prr[3], d = Prr[4];
  const double tr = a + d, half = 0.5 * (a - d), disc = half * half + b * c;
  if (disc < 0.0) { if (ok) *ok = 0; return EKF_OK; }
  const double rt = sqrt(disc);
  double l[2] = {0.5 * tr + rt, 0.5 * tr - rt};
  double v[2][2];
  for (int k = 0; k < 2; ++k) {
    double vx, vy;
    if (b != 0.0) { vx = b; vy = l[k] - a; }
    else if (c != 0.0) { vx = l[k] - d; vy = c; }
    else { vx = ((k == 0) == (a >= d)) ? 1.0 : 0.0; vy = 1.0 - vx; }
    const double nrm = sqrt(vx * vx + vy * vy);
    if (nrm > 0.0) { vx /= nrm; vy /= nrm; }
    v[k][0] = vx; v[k][1] = vy;
  }
  if (fabs(l[1]) < fabs(l[0])) {
    double t = l[0]; l[0] = l[1]; l[1] = t;
    t = v[0][0]; v[0][0] = v[1][0]; v[1][0] = t;
    t = v[0][1]; v[0][1] = v[1][1]; v[1][1] = t;
  }
  for (int k = 0; k < 2; ++k) axii[k] = 2.f * (float)sqrt(5.991 * fabs(l[k]));   /* Robot.cpp:104 */
  *angle = (float)atan2(v[1][0], v[1][1]);                                          /* Robot.cpp:113 */
  if (ok) *ok = 1;
  return EKF_OK;
}

int ekf_download(ekf_ctx* ctx, double* y, double* P, int* n_lines) {
  if (!ctx) return EKF_EINVAL;
  if (ctx->scan_open) { snprintf(ctx->err, sizeof ctx->err, "ekf_download inside an open scan"); return EKF_ESTATE; }
  NOT_POISONED(ctx);
  CU(cudaSetDevice(ctx->cfg.device));
  { int rc = drain(ctx); if (rc) return rc; }
  int rc = read_state(ctx);
  if (rc) return rc;
  const int n = ctx->g.n, nl = 3 + 2 * ctx->h_st->L;
  if (n_lines) *n_lines = ctx->h_st->L;
  if (y) {
    memset(y, 0, (size_t)n * sizeof(double));
    CU(cudaMemcpyAsync(y, ctx->b.y, (size_t)nl * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  if (P) { rc = download_rect(ctx, 0, 0, n, n, P, (size_t)n); if (rc) return rc; }
  return EKF_OK;
}

int ekf_download_live(ekf_ctx* ctx, double* y, double* P, int ldp, int max_n, int* n_lines) {
  if (!ctx) return EKF_EINVAL;
  if (ctx->scan_open) { snprintf(ctx->err, sizeof ctx->err, "ekf_download_live inside an open scan"); return EKF_ESTATE; }
  NOT_POISONED(ctx);
  CU(cudaSetDevice(ctx->cfg.device));
  { int rc = drain(ctx); if (rc) return rc; }
  int rc = read_state(ctx);
  if (rc) return rc;
  const int nl = 3 + 2 * ctx->h_st->L;
  if (n_lines) *n_lines = ctx->h_st->L;
  if (nl > max_n || (P && ldp < nl)) { snprintf(ctx->err, sizeof ctx->err, "live dimension %d exceeds the buffer", nl); return EKF_EINVAL; }
  if (y) {
    CU(cudaMemcpyAsync(y, ctx->b.y, (size_t)nl * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  if (P) { rc = download_rect(ctx, 0, 0, nl, nl, P, (size_t)ldp); if (rc) return rc; }
  return EKF_OK;
}

int ekf_download_block(ekf_ctx* ctx, int r0, int c0, int nr, int nc, double* out) {
  if (!ctx || !out || r0 < 0 || c0 < 0 || nr < 0 || nc < 0 || r0 + nr > ctx->g.n || c0 + nc > ctx->g.n) return EKF_EINVAL;
  if (ctx->scan_open) return EKF_ESTATE;
  CU(cudaSetDevice(ctx->cfg.device));
  { int rc = drain(ctx); if (rc) return rc; }
  return download_rect(ctx, r0, c0, nr, nc, out, (size_t)nc);
}

int ekf_upload(ekf_ctx* ctx, const double* y, const double* P, int n_lines) {
  if (!ctx || n_lines < 0 || n_lines > ctx->g.cap) return EKF_EINVAL;
  if (ctx->scan_open) return EKF_ESTATE;
  CU(cudaSetDevice(ctx->cfg.device));
  { int rc = drain(ctx); if (rc) return rc; }
  const int n = ctx->g.n, nl = 3 + 2 * n_lines;
  int rc = read_state(ctx);
  if (rc) return rc;
  if (y) CU(cudaMemcpyAsync(ctx->b.y, y, (size_t)nl * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  if (P) {
    size_t rows_per = kStageElems / (size_t)nl;
    if (rows_per < 1) rows_per = 1;
    if (rows_per > (size_t)nl) rows_per = nl;
    rc = ensure_stage(ctx, rows_per * (size_t)nl);
    if (rc) return rc;
    for (int r = 0; r < nl; r += (int)rows_per) {
      const int cnt = (nl - r < (int)rows_per) ? nl - r : (int)rows_per;
      CU(cudaMemcpy2DAsync(ctx->d_stage, (size_t)nl * sizeof(double), P + (size_t)r * n, (size_t)n * sizeof(double),
                           (size_t)nl * sizeof(double), cnt, cudaMemcpyHostToDevice, ctx->stream));
      CU(ekf_launch_scatter(ctx->g, ctx->b, r, cnt, nl, ctx->d_stage, nl, ctx->stream));
      CU(cudaStreamSynchronize(ctx->stream));
    }
  }
  /* pose mirrors follow y[0:3] exactly as after an update (Robot.cpp:597-599) */
  EkfDevState s = *ctx->h_st;
  s.L = n_lines;
  if (y) { s.pose[0] = y[0]; s.pose[1] = y[1]; s.pose[2] = y[2]; }
  *ctx->h_st = s;
  CU(cudaMemcpyAsync(ctx->b.st, ctx->h_st, sizeof(EkfDevState), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->L_ub = n_lines;
  ctx->snap_inflight = 0;
  if (y && P) ctx->poisoned = 0;      /* a complete state replaces whatever a failed exchange left behind */
  return EKF_OK;
}

/* Marginalising landmarks out of the Gaussian deletes their entries of y and their rows and columns of P: a gather of
 * the kept entries, no arithmetic.  Hot storage goes through the stage; the cold upper triangle goes out of place into
 * the second covariance buffer when there is one, else in place through the stage in batches of destination rows in
 * increasing order: a later batch reads source rows keep[r] >= r, past every row already written, so the kernel
 * boundaries are the only ordering needed. */
int ekf_remove_lines(ekf_ctx* ctx, int k, const int* lines, int* n_lines) {
  if (!ctx) return EKF_EINVAL;
  if (k < 0 || (k > 0 && !lines)) { snprintf(ctx->err, sizeof ctx->err, "ekf_remove_lines: k = %d, lines = %p", k, (const void*)lines); return EKF_EINVAL; }
  if (ctx->g.world > 1) {
    snprintf(ctx->err, sizeof ctx->err, "ekf_remove_lines: not supported on a row-sharded filter (rows would move between ranks)");
    return EKF_EINVAL;
  }
  if (ctx->scan_open) { snprintf(ctx->err, sizeof ctx->err, "ekf_remove_lines inside an open scan"); return EKF_ESTATE; }
  NOT_POISONED(ctx);
  CU(cudaSetDevice(ctx->cfg.device));
  int rc = read_state(ctx);               /* the exact line count; nothing is changed before the list is validated */
  if (rc) return rc;
  const int L = ctx->h_st->L;
  for (int i = 0; i < k; ++i)
    if (lines[i] < 0 || lines[i] >= L || (i > 0 && lines[i] <= lines[i - 1])) {
      snprintf(ctx->err, sizeof ctx->err, "ekf_remove_lines: lines[%d] = %d (need strictly increasing indices in [0, %d))", i, lines[i], L);
      return EKF_EINVAL;
    }
  if (k == 0) { if (n_lines) *n_lines = L; return EKF_OK; }
  rc = drain(ctx);                        /* no sweep in flight, no open group: Pbuf[rd] is the one complete covariance */
  if (rc) return rc;
  const int Ln = L - k, nl = 3 + 2 * Ln;
  std::vector<int> keep((size_t)nl);
  for (int i = 0; i < 3; ++i) keep[i] = i;
  for (int j = 0, t = 0, jn = 0; j < L; ++j) {
    if (t < k && lines[t] == j) { ++t; continue; }
    keep[3 + 2 * jn] = 3 + 2 * j; keep[4 + 2 * jn] = 4 + 2 * j; ++jn;
  }
  if (!ctx->d_keep) CU(cudaMalloc(&ctx->d_keep, (size_t)ctx->g.n * sizeof(int)));
  CU(cudaMemcpyAsync(ctx->d_keep, keep.data(), (size_t)nl * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  const size_t hot = 6 * (size_t)nl - 6;
  size_t rows_per = kStageElems / (size_t)nl;
  if (rows_per < 1) rows_per = 1;
  if (rows_per > (size_t)nl) rows_per = nl;
  rc = ensure_stage(ctx, hot > rows_per * nl ? hot : rows_per * nl);
  if (rc) return rc;
  CU(ekf_launch_remove_hot(ctx->g, ctx->b, ctx->d_keep, nl, ctx->d_stage, 0, ctx->stream));
  CU(ekf_launch_remove_hot(ctx->g, ctx->b, ctx->d_keep, nl, ctx->d_stage, 1, ctx->stream));
  const size_t ld = ctx->g.ld;
  if (ctx->overlap) {                     /* out of place: Pbuf[rd] -> Pbuf[rd ^ 1], which becomes the line stream's buffer */
    const int dst = ctx->rd ^ 1;
    CU(ekf_launch_remove_cold(ctx->Pbuf[ctx->rd], ld, 0, ctx->Pbuf[dst], ld, 0, ctx->d_keep, 3, nl - 3, nl, 0, ctx->stream));
    ctx->rd = dst;
    ctx->b.P = ctx->Pbuf[ctx->rd];
    ctx->launches += 3;
  } else {
    /* in place: rows and columns before the first removed index keep their place, so rows above it only move their
     * columns from it on */
    const int f = 3 + 2 * lines[0];
    for (int r0 = 3; r0 < nl; r0 += (int)rows_per) {
      const int cnt = nl - r0 < (int)rows_per ? nl - r0 : (int)rows_per;
      CU(ekf_launch_remove_cold(ctx->b.P, ld, 0, ctx->d_stage, (size_t)nl, r0, ctx->d_keep, r0, cnt, nl, f, ctx->stream));
      CU(ekf_launch_remove_cold(ctx->d_stage, (size_t)nl, r0, ctx->b.P, ld, 0, 0, r0, cnt, nl, f, ctx->stream));
      ctx->launches += 2;
    }
    ctx->launches += 2;
  }
  ctx->h_st->L = Ln;
  CU(cudaMemcpyAsync(&ctx->b.st->L, &ctx->h_st->L, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->L_ub = Ln;
  ctx->snap_inflight = 0;
  if (n_lines) *n_lines = Ln;
  return EKF_OK;
}

/* Appending landmarks with no cross-covariance to the rest is y' = [y, lines], P' = [[P, 0], [0, C]]: writes of the new
 * entries, no arithmetic.  After the drain Pbuf[rd] is the one complete covariance and every later path reads from it or
 * from a sweep that writes every live element of its destination, so only Pbuf[rd] is written (DESIGN section 3.3). */
int ekf_insert_lines(ekf_ctx* ctx, int k, const double* lines, const double* cov, int* n_lines) {
  if (!ctx) return EKF_EINVAL;
  if (k < 0 || (k > 0 && !lines)) { snprintf(ctx->err, sizeof ctx->err, "ekf_insert_lines: k = %d, lines = %p", k, (const void*)lines); return EKF_EINVAL; }
  for (int i = 0; i < 2 * k; ++i)
    if (!isfinite(lines[i])) { snprintf(ctx->err, sizeof ctx->err, "ekf_insert_lines: lines[%d] = %g is not finite", i, lines[i]); return EKF_EINVAL; }
  const size_t w = 2 * (size_t)k;
  if (cov) {
    for (size_t i = 0; i < w; ++i)
      if (!(cov[i * w + i] >= 0.0)) {
        snprintf(ctx->err, sizeof ctx->err, "ekf_insert_lines: cov[%zu][%zu] = %g (need a finite, non-negative diagonal)", i, i, cov[i * w + i]);
        return EKF_EINVAL;
      }
    /* the upper triangle against the lower one in 64 x 64 tiles: the transposed reads stay in cache */
    const size_t T = 64;
    for (size_t i0 = 0; i0 < w; i0 += T)
      for (size_t c0 = i0; c0 < w; c0 += T)
        for (size_t i = i0; i < i0 + T && i < w; ++i)
          for (size_t c = c0 > i ? c0 : i; c < c0 + T && c < w; ++c)
            if (!isfinite(cov[i * w + c]) || cov[i * w + c] != cov[c * w + i]) {
              snprintf(ctx->err, sizeof ctx->err, "ekf_insert_lines: cov[%zu][%zu] = %g is not finite or not symmetric", i, c, cov[i * w + c]);
              return EKF_EINVAL;
            }
  }
  if (ctx->g.world > 1) {
    snprintf(ctx->err, sizeof ctx->err, "ekf_insert_lines: not supported on a row-sharded filter");
    return EKF_EINVAL;
  }
  if (ctx->scan_open) { snprintf(ctx->err, sizeof ctx->err, "ekf_insert_lines inside an open scan"); return EKF_ESTATE; }
  NOT_POISONED(ctx);
  CU(cudaSetDevice(ctx->cfg.device));
  int rc = read_state(ctx);               /* the exact line count; nothing is changed before the capacity is checked */
  if (rc) return rc;
  const int L = ctx->h_st->L;
  if ((long long)L + k > ctx->g.cap) {
    snprintf(ctx->err, sizeof ctx->err, "ekf_insert_lines: %d + %d landmarks exceed the capacity of %d (nothing was inserted)", L, k, ctx->g.cap);
    return EKF_ECAPACITY;
  }
  if (k == 0) { if (n_lines) *n_lines = L; return EKF_OK; }
  rc = drain(ctx);                        /* no sweep in flight, no open group: Pbuf[rd] is the one complete covariance */
  if (rc) return rc;
  const int nl_old = 3 + 2 * L, nl = nl_old + 2 * k;
  std::vector<double> hot((size_t)5 * k);
  for (int e = 0; e < k; ++e) {
    const size_t a = 2 * (size_t)e;
    hot[5 * e] = lines[a]; hot[5 * e + 1] = lines[a + 1];
    hot[5 * e + 2] = cov ? cov[a * w + a] : 0.0;
    hot[5 * e + 3] = cov ? cov[a * w + a + 1] : 0.0;
    hot[5 * e + 4] = cov ? cov[(a + 1) * w + a + 1] : 0.0;
  }
  size_t rows_per = kStageElems / w;
  if (rows_per > w) rows_per = w;
  rc = ensure_stage(ctx, hot.size() > rows_per * w ? hot.size() : rows_per * w);
  if (rc) return rc;
  CU(cudaMemcpyAsync(ctx->d_stage, hot.data(), hot.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  CU(ekf_launch_insert_hot(ctx->g, ctx->b, L, k, ctx->d_stage, ctx->stream));
  const size_t ld = ctx->g.ld;
  /* the rows above the new block: 2k zeros each (and, surveyed, the new rows too) */
  CU(ekf_launch_insert_cold(ctx->b.P, ld, nl_old, nl, 3, (cov ? nl_old : nl) - 3, 0, 0, ctx->stream));
  ctx->launches += 2;
  if (cov) {
    for (size_t i0 = 0; i0 < w; i0 += rows_per) {
      const size_t cnt = w - i0 < rows_per ? w - i0 : rows_per;
      CU(cudaMemcpyAsync(ctx->d_stage, cov + i0 * w, cnt * w * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
      CU(ekf_launch_insert_cold(ctx->b.P, ld, nl_old, nl, nl_old + (int)i0, (int)cnt, ctx->d_stage, (int)i0, ctx->stream));
      CU(cudaStreamSynchronize(ctx->stream));
      ctx->launches++;
    }
  }
  ctx->h_st->L = L + k;
  CU(cudaMemcpyAsync(&ctx->b.st->L, &ctx->h_st->L, sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->L_ub = L + k;
  ctx->snap_inflight = 0;
  if (n_lines) *n_lines = L + k;
  return EKF_OK;
}

/* An absolute pose fix is a rank-d (d <= 3) update whose gain needs only P[:, 0:3], which is hot storage and current at
 * all times.  The call drains first (no open sweep group, no sweep in flight: Pbuf[rd] is the one complete covariance),
 * then enqueues the gain, the hot update and one in-place sweep of (at most) two rank-2 terms.  A rejected fix or a
 * singular S leaves st->np = 0, and every sweep form returns without writing for a zero count: the state is unchanged. */
int ekf_observe_pose(ekf_ctx* ctx, int mask, const double z[3], const double R[9], double d2_max, double* d2,
                     int* accepted, double pose[3]) {
  if (!ctx) return EKF_EINVAL;
  if (mask < 1 || mask > 7 || !z || !R || d2_max != d2_max) {
    snprintf(ctx->err, sizeof ctx->err, "ekf_observe_pose: mask = %d, z = %p, R = %p, d2_max = %g", mask, (const void*)z,
             (const void*)R, d2_max);
    return EKF_EINVAL;
  }
  EkfPoseFix f;
  memset(&f, 0, sizeof f);
  int d = 0;
  for (int c = 0; c < 3; ++c) if (mask & (1 << c)) f.sel[d++] = c;
  for (int i = 0; i < d; ++i) {
    f.z[i] = z[f.sel[i]];
    if (!isfinite(f.z[i])) { snprintf(ctx->err, sizeof ctx->err, "ekf_observe_pose: z[%d] is not finite", f.sel[i]); return EKF_EINVAL; }
    for (int k = 0; k < d; ++k) {
      const int r = f.sel[i], c = f.sel[k];
      f.R[3 * i + k] = R[3 * r + c];
      if (!isfinite(R[3 * r + c]) || R[3 * r + c] != R[3 * c + r]) {
        snprintf(ctx->err, sizeof ctx->err, "ekf_observe_pose: R[%d][%d] = %g is not finite or not symmetric", r, c, R[3 * r + c]);
        return EKF_EINVAL;
      }
    }
  }
  f.d2max = d2_max;
  if (ctx->g.world > 1) {
    snprintf(ctx->err, sizeof ctx->err, "ekf_observe_pose: not supported on a row-sharded filter");
    return EKF_EINVAL;
  }
  if (ctx->scan_open) { snprintf(ctx->err, sizeof ctx->err, "ekf_observe_pose inside an open scan"); return EKF_ESTATE; }
  NOT_POISONED(ctx);
  CU(cudaSetDevice(ctx->cfg.device));
  int rc = drain(ctx);
  if (rc) return rc;
  /* term 2 goes to slot 1; with a single slot (max_batch = 1) to a scratch row, folded by a second one-term sweep */
  const bool one_slot = ctx->slots < 2;
  const size_t ld = ctx->g.ld;
  if (one_slot) { rc = ensure_stage(ctx, 4 * ld); if (rc) return rc; }
  double2* K2 = one_slot ? (double2*)ctx->d_stage : ctx->b.Kp + ld;
  double2* KS2 = one_slot ? (double2*)ctx->d_stage + ld : ctx->b.KSp + ld;
  CU(ekf_launch_pose_gain(ctx->g, ctx->b, f, d, K2, KS2, ctx->L_ub, ctx->stream));
  CU(ekf_launch_pose_apply(ctx->g, ctx->b, d, K2, KS2, one_slot ? 1 : 2, ctx->L_ub, ctx->stream));
  ctx->launches += 2;
  rc = sweep_now(ctx, (d == 3 && !one_slot) ? 2 : 1);
  if (rc) return rc;
  if (one_slot && d == 3) {
    CU(ekf_launch_pose_term2(ctx->g, ctx->b, d, K2, KS2, ctx->L_ub, ctx->stream));
    ctx->launches++;
    rc = sweep_now(ctx, 1);
    if (rc) return rc;
  }
  if (!d2 && !accepted && !pose) return EKF_OK;
  rc = read_state(ctx);
  if (rc) return rc;
  const int st = ctx->h_st->fix_status;
  if (d2) *d2 = ctx->h_st->fix_d2;
  if (accepted) *accepted = st == EKF_FIX_ACCEPTED;
  if (pose) memcpy(pose, ctx->h_st->pose, 3 * sizeof(double));
  if (st == EKF_FIX_SINGULAR) {
    snprintf(ctx->err, sizeof ctx->err, "ekf_observe_pose: S is singular (mask %d); the state is unchanged", mask);
    return EKF_ESINGULAR;
  }
  return EKF_OK;
}

int ekf_cov_stats(ekf_ctx* ctx, double* trace, double* sum, double* sumsq) {
  if (!ctx) return EKF_EINVAL;
  if (ctx->scan_open) return EKF_ESTATE;
  CU(cudaSetDevice(ctx->cfg.device));
  { int rc = drain(ctx); if (rc) return rc; }
  CU(ekf_launch_cov_stats(ctx->g, ctx->b, ctx->d_partials, ctx->g.n, ctx->d_out3, ctx->stream));
  double o[3];
  CU(cudaMemcpyAsync(o, ctx->d_out3, sizeof o, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  if (trace) *trace = o[0];
  if (sum) *sum = o[1];
  if (sumsq) *sumsq = o[2];
  return EKF_OK;
}

/* ------------------------------------------ measurement ------------------------------------------ */
int ekf_profile_enable(ekf_ctx* ctx, int on) {
  if (!ctx) return EKF_EINVAL;
  ctx->prof = on ? 1 : 0;
  ctx->ev_used = 0; ctx->ev_bytes.clear(); ctx->lev_used = 0;
  return EKF_OK;
}

int ekf_profile_read(ekf_ctx* ctx, int* n_sweeps, double* sweep_ms, double* sweep_bytes, long long* launches) {
  if (!ctx) return EKF_EINVAL;
  CU(cudaSetDevice(ctx->cfg.device));
  if (ctx->wstream) CU(cudaStreamSynchronize(ctx->wstream));
  int rc = read_state(ctx);
  if (rc) return rc;
  const double n = 3.0 + 2.0 * ctx->h_st->L;
  double ms = 0.0, bytes = 0.0;
  const size_t ns = ctx->ev_used / 2;
  for (size_t i = 0; i < ns; ++i) {
    float t = 0.f;
    CU(cudaEventElapsedTime(&t, ctx->ev[2 * i], ctx->ev[2 * i + 1]));
    ms += t;
    bytes += 8.0 * n * (n + 1.0) + 32.0 * n * ctx->ev_bytes[i];     /* SURVEY 8d: B_sweep(n, m) */
  }
  if (n_sweeps) *n_sweeps = (int)ns;
  if (sweep_ms) *sweep_ms = ms;
  if (sweep_bytes) *sweep_bytes = bytes;
  if (launches) *launches = ctx->launches;
  ctx->ev_used = 0; ctx->ev_bytes.clear(); ctx->launches = 0;
  return EKF_OK;
}

int ekf_profile_read_lines(ekf_ctx* ctx, int* n_scans, double* line_ms) {
  if (!ctx) return EKF_EINVAL;
  CU(cudaSetDevice(ctx->cfg.device));
  CU(cudaStreamSynchronize(ctx->stream));
  double ms = 0.0;
  const size_t ns = ctx->lev_used / 2;
  for (size_t i = 0; i < ns; ++i) {
    float t = 0.f;
    CU(cudaEventElapsedTime(&t, ctx->lev[2 * i], ctx->lev[2 * i + 1]));
    ms += t;
  }
  if (n_scans) *n_scans = (int)ns;
  if (line_ms) *line_ms = ms;
  ctx->lev_used = 0;
  return EKF_OK;
}

int ekf_timer_start(ekf_ctx* ctx) {
  if (!ctx) return EKF_EINVAL;
  CU(cudaSetDevice(ctx->cfg.device));
  if (!ctx->t0) { CU(cudaEventCreate(&ctx->t0)); CU(cudaEventCreate(&ctx->t1)); }
  CU(cudaEventRecord(ctx->t0, ctx->stream));
  return EKF_OK;
}

int ekf_timer_stop(ekf_ctx* ctx, double* ms) {
  if (!ctx || !ctx->t0) return EKF_EINVAL;
  CU(cudaSetDevice(ctx->cfg.device));
  if (ctx->overlap) {          /* the sweeps in flight belong to the timed work, and so does the sweep of the open group */
    { int rc = close_group(ctx); if (rc) return rc; }
    for (int p = 0; p < 2; ++p) if (ctx->evF_used[p]) CU(cudaStreamWaitEvent(ctx->stream, ctx->evF[p], 0));
  }
  CU(cudaEventRecord(ctx->t1, ctx->stream));
  CU(cudaEventSynchronize(ctx->t1));
  float t = 0.f;
  CU(cudaEventElapsedTime(&t, ctx->t0, ctx->t1));
  if (ms) *ms = (double)t;
  return EKF_OK;
}

int ekf_sweep_probe(ekf_ctx* ctx, int m, int repeats, double* ms_each) {
  if (!ctx || m < 1 || m > ctx->cfg.max_batch || repeats < 1) return EKF_EINVAL;
  if (ctx->scan_open) return EKF_ESTATE;
  CU(cudaSetDevice(ctx->cfg.device));
  { int rc = drain(ctx); if (rc) return rc; }
  CU(ekf_launch_zero_pending(ctx->g, ctx->b, m, &ctx->b.st->np, ctx->stream));
  { int rc = launch_sweep(ctx, m); if (rc) return rc; }                        /* warm-up */
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  CU(cudaEventRecord(e0, ctx->stream));
  for (int i = 0; i < repeats; ++i) { int rc = launch_sweep(ctx, m); if (rc) return rc; }
  CU(cudaEventRecord(e1, ctx->stream));
  CU(cudaMemsetAsync(&ctx->b.st->np, 0, sizeof(int), ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  float t = 0.f;
  CU(cudaEventElapsedTime(&t, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  if (ms_each) *ms_each = (double)t / repeats;
  return EKF_OK;
}

}  /* extern "C" */
