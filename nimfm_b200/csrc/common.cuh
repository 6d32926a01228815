// common.cuh -- private structures and helpers of libnimfm_cuda.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <initializer_list>
#include <string>
#include <vector>

#include "../../include/nimfm_cuda.h"

struct ncclComm;

#define NIMFM_MAX_DEGREE 6   // device row kernels are instantiated for degree 2..6
#define NIMFM_MAX_RANKS 8    // ranks the peer-memory exchange is instantiated for (one NVSwitch box)

struct nimfm_ctx {
  int device = 0;
  int numSMs = 0;
  int smemOptin = 0;          // max opt-in dynamic shared memory per block
  int smemPerSM = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::string err;
  int64_t launches = 0;
  // scratch (grown on demand)
  double *partials = nullptr;  // per-group partial sums written by the row kernels
  size_t partialsCap = 0;
  double *stash = nullptr;     // deterministic gradient (fm_cols.cu): per-row stash records + segment partials
  size_t stashCap = 0;
  struct nimfm_mb_index *mbIndex = nullptr;   // deterministic AdaGrad: the column index of the current minibatch
  double *scalars = nullptr;  // small device scalar block (64 doubles)
  double *hostScalars = nullptr;  // pinned mirror
  int64_t *idxScratch = nullptr;  // device copy of host-provided row ids
  size_t idxCap = 0;
  int32_t *idx32Scratch = nullptr;
  // host-streaming staging (nimfm_fm_loss_grad_host): two buffer sets + a copy stream
  cudaStream_t copyStream = nullptr;
  cudaEvent_t evCopied[2] = {nullptr, nullptr}, evComputed[2] = {nullptr, nullptr};
  cudaEvent_t tev0 = nullptr, tev1 = nullptr;   // nimfm_timer_*
  struct Stage {
    double *packed = nullptr;      // packed transport of the values (host_stage.h, pack_values): expanded into data
    uint64_t *mask = nullptr;
    uint32_t *blk = nullptr;
    size_t capPack = 0;
    double *data = nullptr, *y = nullptr;
    int64_t *idx64 = nullptr, *indptr = nullptr;
    int32_t *idx32 = nullptr;
    size_t capNnz = 0, capRows = 0, capIdx64 = 0;
  } stage[2];
  // pinned slots of the host staging team (host_stage.h): narrowed ids + rebased indptr
  int32_t *hostIdx[4] = {nullptr, nullptr, nullptr, nullptr};
  int64_t *hostPtr[4] = {nullptr, nullptr, nullptr, nullptr};
  double *hostPack[4] = {nullptr, nullptr, nullptr, nullptr};   // packed values: pinned slots of the staging team
  uint64_t *hostMask[4] = {nullptr, nullptr, nullptr, nullptr};
  uint32_t *hostBlk[4] = {nullptr, nullptr, nullptr, nullptr};
  size_t hostCapPack = 0;
  double *hostData[4] = {nullptr, nullptr, nullptr, nullptr};   // pageable callers only: values / targets
  double *hostY[4] = {nullptr, nullptr, nullptr, nullptr};
  size_t hostCapData = 0, hostCapY = 0;
  int32_t lastPageable = 0;          // nimfm_stream_stats: the last host-fed call staged pageable values
  cudaEvent_t evSlot[4] = {nullptr, nullptr, nullptr, nullptr};
  size_t hostCapNnz = 0, hostCapRows = 0;
  // pinned pieces of the file -> device copy (loaders.cu, staged_h2d): kPinPieces x kPinPieceBytes
  static constexpr int kPinPieces = 16;
  static constexpr size_t kPinPieceBytes = 8u << 20;
  unsigned char *pinPiece[kPinPieces] = {nullptr};
  cudaEvent_t evPiece[kPinPieces] = {nullptr};
  int64_t lastH2D = 0, lastD2H = 0;   // nimfm_stream_stats
  int32_t lastHostThreads = 0;
  uint8_t *stageHotSlot = nullptr;   // persistent [stageHotD] table; only the <=16 hot entries change per call
  int32_t *stageHotList = nullptr;
  int64_t stageHotD = -1;
  int stageNHot = 0;
  int32_t stagePrevHot[16] = {0};
  // communicator
  ncclComm *comm = nullptr;
  int rank = 0, nranks = 1;
  // NVLink peer memory (peer.cu): buffers that take part in the gradient exchange live in arenas whose IPC
  // handles every rank has opened; arenas are recycled by size and released with the context
  struct PeerArena {
    double *base = nullptr;
    size_t nDoubles = 0;
    bool inUse = false, haveHandle = false;
    int64_t handle[8] = {0};                     // cudaIpcMemHandle_t of base
  };
  struct PeerOpened {                            // a peer's arena this rank has mapped (cached by handle)
    int rank = 0;
    int64_t handle[8] = {0};
    double *ptr = nullptr;
  };
  struct PeerMap {                               // one buffer of the running epoch call: every rank's copy
    double *local = nullptr;
    int64_t nDoubles = 0;
    double *peer[NIMFM_MAX_RANKS] = {nullptr};
  };
  std::vector<PeerArena> arenas;
  std::vector<PeerOpened> peerOpened;
  std::vector<PeerMap> peerMaps;
  bool peerOK = false;
  uint32_t *peerFlags = nullptr;                 // [NIMFM_MAX_RANKS] arrival counters written by the peers
  uint32_t *peerFlagsOf[NIMFM_MAX_RANKS] = {nullptr};
  uint32_t barrierEpoch = 0;
  // NIMFM_TRACE=1: device time per phase of the multi-rank epochs (CUDA events on the stream, summed per tag and
  // printed to stderr by nimfm_trace_report) -- a measurement aid, off by default
  struct TraceSpan { const char *tag; cudaEvent_t e0, e1; bool open; };   // spans may nest: end closes the innermost
  std::vector<TraceSpan> trace;
  int traceOn = -1;
};
void nimfm_trace_begin(nimfm_ctx *ctx, const char *tag);
void nimfm_trace_end(nimfm_ctx *ctx);
void nimfm_trace_report(nimfm_ctx *ctx, const char *what);
struct TraceReport {   // reports (and releases) the spans recorded since the last report on every exit path
  nimfm_ctx *ctx;
  const char *what;
  bool on;
  ~TraceReport() { if (on) nimfm_trace_report(ctx, what); }
};

struct nimfm_dataset;
// fm_cols.cu: the CSC twin of a CSR dataset (stable transpose: rows ascending inside a column) and its columns cut
// into segments of at most 512 entries -- the work list of the column-wise (atomic-free) gradient kernels
struct nimfm_det_twin {
  nimfm_dataset *csc = nullptr;
  int32_t *taskCol = nullptr, *taskLen = nullptr, *taskSlot = nullptr;   // per segment: column, length, partial slot (-1: whole column)
  int64_t *taskBeg = nullptr;
  int32_t *multiCol = nullptr, *multiFirst = nullptr, *multiCount = nullptr;   // columns with several segments
  int64_t nTasks = 0, nMulti = 0, nSlots = 0;
  int nAug = -1;
};
void nimfm_det_twin_free(nimfm_ctx *ctx, nimfm_det_twin *t);
int nimfm_det_twin_get(nimfm_ctx *ctx, const nimfm_dataset *X, int nAug, nimfm_det_twin **out);

struct nimfm_dataset {
  int kind = NIMFM_DS_CSR;
  mutable nimfm_det_twin *detTwin = nullptr;
  int64_t n = 0, d = 0, nnz = 0;     // n rows (samples), d columns (features) of the LOGICAL matrix
  int64_t nFields = 0;
  int64_t maxSegNnz = 0;             // longest row (CSR) / column (CSC)
  double *data = nullptr;
  int32_t *indices = nullptr;        // column ids (CSR) / row ids (CSC), narrowed to int32
  int64_t *indptr = nullptr;
  int32_t *fields = nullptr;
  mutable int fieldDup = -1;         // field datasets: does a row repeat a field? (-1 = not checked yet; ffm.cu)
  double *y = nullptr;
  // hot features (CSR kinds): columns present in >= 1/16 of a row sample, at most 16 (fm_rows.cuh)
  uint8_t *hotSlot = nullptr;        // [d], 255 = cold
  int32_t *hotList = nullptr;        // [nHot]
  int nHot = 0;
  // CD only: runs of consecutive columns with pairwise-disjoint row support (built at cd_begin)
  std::vector<int64_t> cdBatchStart;
};

// dataset_ops.cu: buffers of the stable sort behind nimfm_dataset_transpose, owned by the caller
struct TransposeScratch {
  int32_t *segOf, *keysOut;
  uint32_t *permIn, *permOut;
  void *tmp;          // CUB scratch; nullptr: nimfm_transpose_sort only sets tmpBytes
  size_t tmpBytes;
};
int nimfm_transpose_sort(nimfm_ctx *ctx, int64_t nsIn, int64_t nsOut, int64_t nnz, const int64_t *inPtr,
                         const int32_t *inIdx, const double *inData, TransposeScratch *s, double *outData,
                         int32_t *outIdx, int64_t *outPtr);

// dataset_ops.cu: the column index of ONE minibatch (rows rowIdx[0 .. B), or (rowBegin + q) mod n for q < B: a
// cursor that may wrap past the last row, and pass it more than once when B > n), built on the device for the
// deterministic minibatch solvers (AdaGrad, MBPSGD, minibatch SGD).  view: the B rows gathered into a CSR (CSR-field)
// dataset that keeps the parent's d, nFields, maxSegNnz, hot table and field-repeat flag; csc: its stable
// column-major twin, whose indices are positions 0 .. B-1 in the view (a row listed twice gives two positions); tw:
// that twin's 512-entry segments in the dataset twin's layout (dummy columns d + a span all B positions).  Held by the
// context, grown on demand, rebuilt per minibatch; view, csc and tw only point into the buffers below.
struct nimfm_mb_index {
  nimfm_dataset view, csc;
  nimfm_det_twin tw;
  double *bias = nullptr;   // [1]: the intercept the minibatch's forward pass sees (AdaGrad refreshes it from g_sum)
  int64_t *rows = nullptr, *rowLen = nullptr, *ptr = nullptr, *cPtr = nullptr, *colCnt = nullptr, *tot = nullptr;
  int64_t *hostTot = nullptr;   // pinned: entries, tasks, multi-segment columns, partial slots
  double *data = nullptr, *y = nullptr, *cData = nullptr;
  double *yhat = nullptr;       // [B] scratch for the forward pass's decision values
  int32_t *idx = nullptr, *fld = nullptr, *cIdx = nullptr, *segOf = nullptr, *keysOut = nullptr;
  uint32_t *permIn = nullptr, *permOut = nullptr;
  unsigned char *tmp = nullptr;
  long long *segOff = nullptr;   // per-column segment counts and their exclusive scan
  int32_t *taskCol = nullptr, *taskLen = nullptr, *taskSlot = nullptr, *multiCol = nullptr, *multiFirst = nullptr,
          *multiCount = nullptr;
  int64_t *taskBeg = nullptr;
  size_t capRows = 0, capRowLen = 0, capPtr = 0, capY = 0, capCol = 0, capColPtr = 0, capSeg = 0, capTot = 0,
         capBias = 0, capYhat = 0, capTmp = 0, capData = 0, capIdx = 0, capCData = 0, capCIdx = 0, capSegOf = 0, capKeys = 0,
         capPermIn = 0, capPermOut = 0, capFld = 0, capTaskCol = 0, capTaskBeg = 0, capTaskLen = 0, capTaskSlot = 0,
         capMultiCol = 0, capMultiFirst = 0, capMultiCount = 0;
};
int nimfm_mb_index_build(nimfm_ctx *ctx, const nimfm_dataset *X, int nAug, int64_t rowBegin, int64_t nRows,
                         const int32_t *rowIdx, nimfm_mb_index **out);
void nimfm_mb_index_free(nimfm_mb_index *m);

struct nimfm_fm {
  int degree = 2, k = 1, nOrders = 1, nAug = 0;
  int64_t d = 0;           // nFeatures (without dummies)
  int fitLinear = 1, fitIntercept = 1;
  int64_t dd() const { return d + nAug; }
  int64_t nP() const { return (int64_t)nOrders * dd() * k; }
  // device parameters, layout P[j][o][s] ("feature-major": one feature's nOrders*k doubles contiguous).
  // P, w and the scalar block b live in ONE allocation, pool = [P (nP) | w (d) | b (8) | slack], in the same flat
  // element order as the gradient buffer, so that a multi-rank step can reduce-scatter the gradients, update
  // its flat slice of the parameters and all-gather the pool in place (fm_api.cu, sharded MBPSGD step).
  double *pool = nullptr;
  int64_t poolCap = 0;     // doubles allocated in pool and in grad (>= nP + d + 8, plus slice-alignment slack)
  double *P = nullptr, *w = nullptr, *lams = nullptr;
  double *b = nullptr;     // device scalar block inside pool: [0]=intercept, [1]=epoch loss of the sharded step
  bool lamsAreOnes = true;
  // gradient buffer: [gP (nP) | gw (d) | gb, lossSum | slack] contiguous for a single collective
  double *grad = nullptr;
  double *proxState = nullptr;   // SquaredL12 column prox: [tau | prevCnt | settled | done] (prox_kernels.cuh)
  // lazy MBPSGD epoch: per-feature {1/cumP, 1/cumW} at the feature's last update, touched flags
  double2 *lazyInv = nullptr;
  uint8_t *lazyFlag = nullptr;
  // AdaGrad state (same layouts): g_sum, g_norm, and per-minibatch deltas
  double *gsP = nullptr, *gnP = nullptr, *gsw = nullptr, *gnw = nullptr;
  double *dG = nullptr;    // [dGsP (nP) | dGnP (nP) | dGsw (d) | dGnw (d) | touched (d+nAug) | loss, sum dL, sum dL^2, viol]
  double *adaScal = nullptr;   // device: [gsb, gnb]
  bool adaReady = false;
  // SGD lazy-scaling caches
  double *scalingsP = nullptr, *scalingsW = nullptr, *sgdScal = nullptr;  // sgdScal: [scaling_P, scaling_w, viol, loss]
  bool sgdReady = false;
  double *sgdCnt = nullptr;    // minibatch SGD (sgd_mb.cu): per-feature touch counts of the current minibatch
  double *psgdThr = nullptr;   // PSGD: per-feature accumulated thresholds of the lazy L1 / L21 protocol (psgd.cu)
  bool psgdReady = false;
  // CD caches
  double *Pcm = nullptr;       // component-major copy P[o][s][j] used by the column kernels
  double *yPred = nullptr, *Acache = nullptr, *colNormSq = nullptr, *cdScal = nullptr;
  int64_t cdN = 0;
  bool cdReady = false;
  // reusable host staging
  std::vector<double> hostTmp;
};

struct nimfm_ffm {
  int k = 1;
  int64_t nFields = 0, d = 0;
  int fitLinear = 1, fitIntercept = 1;
  int64_t nP() const { return nFields * d * k; }
  // device layout P[j][f][s]: one feature's nFields*k doubles contiguous
  double *P = nullptr, *w = nullptr, *b = nullptr;
  double *PT = nullptr;        // field-major copy PT[f][j][s], refreshed by the column gradient route (ffm_cols.cuh)
  double *grad = nullptr;      // [gP | gw | gb, lossSum]
  double *gsP = nullptr, *gnP = nullptr, *gsw = nullptr, *gnw = nullptr, *dG = nullptr, *adaScal = nullptr;
  double *sgdCnt = nullptr;    // minibatch SGD (sgd_mb.cu)
  mutable unsigned char *unitScratch = nullptr;   // ffm_units_kernel's records of long rows (ffm.cu), grown on demand
  mutable size_t unitScratchBytes = 0;
  bool adaReady = false;
  double *scalingsP = nullptr, *scalingsW = nullptr, *sgdScal = nullptr;
  bool sgdReady = false;
  std::vector<double> hostTmp;
};

// the lane-group width KT in {4, 8, 16, 32} of a runtime-k kernel that maps lane <-> component (ffm_units_kernel,
// fm_cols_grad_generic_kernel): the one that idles the fewest lanes over ceil(k / KT) component chunks; ties go to
// the wider group (fewer chunks)
inline int lane_group_kt(int k) {
  int best = 32;
  for (int kt = 16; kt >= 4; kt >>= 1)
    if ((int64_t)(k + kt - 1) / kt * kt < (int64_t)(k + best - 1) / best * best) best = kt;
  return best;
}

// ------------------------------------------------------------------ error plumbing
int nimfm_fail(nimfm_ctx *ctx, int code, const char *fmt, ...);

#define CK(call)                                                                             \
  do {                                                                                       \
    cudaError_t e_ = (call);                                                                 \
    if (e_ != cudaSuccess)                                                                   \
      return nimfm_fail(ctx, NIMFM_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call,      \
                        cudaGetErrorString(e_));                                             \
  } while (0)

#define REQUIRE(cond, ...)                                                \
  do {                                                                    \
    if (!(cond)) return nimfm_fail(ctx, NIMFM_ERR_INVALID, __VA_ARGS__);  \
  } while (0)

#define LAUNCHED(ctx) ((ctx)->launches++)

int nimfm_ensure_partials(nimfm_ctx *ctx, size_t nDoubles);
int nimfm_ensure_idx(nimfm_ctx *ctx, size_t n);
int nimfm_allreduce_sum(nimfm_ctx *ctx, double *buf, int64_t n);
int nimfm_reduce_scatter_sum(nimfm_ctx *ctx, double *buf, int64_t count);
int nimfm_allgather_inplace(nimfm_ctx *ctx, double *buf, int64_t count);
int nimfm_allgather_host_i64(nimfm_ctx *ctx, const int64_t *mine, int count, int64_t *all);
// Minibatch schedule shared by the ranks of a synchronous epoch.  Every rank feeds up to `mb` of its own
// `nRows` rows per minibatch; shards and shares may be uneven, so all ranks run T = max_r ceil(nRows_r / mb_r)
// minibatches (a rank that has run out feeds 0 rows but still joins the collectives) and the iteration
// counter advances by the GLOBAL number of rows of the minibatch.
struct MbSchedule {
  int64_t T = 0;
  int rank = 0;
  std::vector<int64_t> nRows, mb;
  int64_t rows_of(int r, int64_t t) const {
    const int64_t left = nRows[(size_t)r] - t * mb[(size_t)r];
    return left <= 0 ? 0 : (left < mb[(size_t)r] ? left : mb[(size_t)r]);
  }
  int64_t local(int64_t t) const { return rows_of(rank, t); }
  int64_t global(int64_t t) const {
    int64_t g = 0;
    for (size_t r = 0; r < nRows.size(); r++) g += rows_of((int)r, t);
    return g;
  }
};
// gathers (nRows, mb, it) of every rank; fails when the ranks disagree on `it` (their replicas have diverged)
int nimfm_mb_schedule(nimfm_ctx *ctx, int64_t nRows, int64_t mb, int64_t it, MbSchedule *out);
// peer.cu
int nimfm_peer_init(nimfm_ctx *ctx);
void nimfm_peer_shutdown(nimfm_ctx *ctx);
int nimfm_comm_alloc(nimfm_ctx *ctx, double **out, size_t nDoubles);   // local; arena memory when peer memory is on
void nimfm_comm_free(nimfm_ctx *ctx, double *p);
int nimfm_peer_prepare(nimfm_ctx *ctx, const double *const *bufs, int nb);   // COLLECTIVE, per epoch-level call
void nimfm_peer_release(nimfm_ctx *ctx);
struct PeerScope {   // prepare on entry, release on every exit path
  nimfm_ctx *ctx;
  int rc;
  PeerScope(nimfm_ctx *c, std::initializer_list<const double *> bufs) : ctx(c), rc(0) {
    bool any = false;   // no buffer to exchange (e.g. allreduce = 0): not a collective call, nothing to prepare
    for (const double *b : bufs) any = any || b != nullptr;
    if (c->nranks > 1 && any) rc = nimfm_peer_prepare(c, bufs.begin(), (int)bufs.size());
  }
  ~PeerScope() { nimfm_peer_release(ctx); }
};
int nimfm_peer_allreduce_sum(nimfm_ctx *ctx, double *buf, int64_t n, int *done);
struct MbpsgdStepArgs {   // Params.step (params.nim:90-98) + L1 prox on a flat slice of [P | w | b, epochLoss]
  int64_t nP, d;
  double negEtaP, rP, lam, negEtaW, rW, negEtaB, rB;
  int reg, fitLinear, fitIntercept;
};
// barrier, then reduce this rank's slice [lo, hi) of `grad` over all ranks (rank order) and step the local `pool`
// there; the caller follows with [prox on the slice,] barrier, nimfm_peer_pull_slices(pool).  *done = 0 when the
// buffers are not peer-mapped (nothing was launched)
int nimfm_peer_mbpsgd_step(nimfm_ctx *ctx, double *pool, double *grad, int64_t lo, int64_t hi, const MbpsgdStepArgs &sa,
                           int *done);
int nimfm_peer_pull_slices(nimfm_ctx *ctx, double *buf, int64_t c, int64_t n);
int nimfm_peer_barrier(nimfm_ctx *ctx);

// hot-column table upload (dataset.cu)
int nimfm_upload_hot(nimfm_ctx *ctx, const std::vector<int32_t> &hot, int64_t d, uint8_t **hotSlot, int32_t **hotList);
int nimfm_staged_h2d(nimfm_ctx *ctx, void *dDst, const void *src, size_t bytes, int64_t narrowD = 0, int *bad = nullptr);
int nimfm_staged_d2h(nimfm_ctx *ctx, void *hostDst, const void *dSrc, size_t bytes);
int nimfm_find_hot(const int64_t *indices, const int64_t *indptr, int64_t rowBegin, int64_t rowEnd,
                   std::vector<int32_t> &hot, int64_t maxSample, int64_t d);

// upload host int64 row ids into ctx->idx32Scratch as int32 (validated against n)
int nimfm_stage_row_ids(nimfm_ctx *ctx, const int64_t *ids, int64_t count, int64_t n);

// ------------------------------------------------------------------ device helpers
#ifdef __CUDACC__

__device__ __forceinline__ double dev_loss(int kind, double thr, double y, double p) {
  switch (kind) {
    case NIMFM_LOSS_SQUARED: { double z = y - p; return 0.5 * (z * z); }
    case NIMFM_LOSS_SQUARED_HINGE: { double z = fmax(1.0 - p * y, 0.0); return z * z; }
    case NIMFM_LOSS_LOGISTIC: {
      double z = p * y;
      return z > 0 ? log(1.0 + exp(-z)) : log(exp(z) + 1.0) - z;
    }
    default: {
      double z = fabs(y - p);
      return z < thr ? 0.5 * (z * z) : thr * (z - 0.5 * thr);
    }
  }
}

__device__ __forceinline__ double dev_dloss(int kind, double thr, double y, double p) {
  switch (kind) {
    case NIMFM_LOSS_SQUARED: return p - y;
    case NIMFM_LOSS_SQUARED_HINGE: { double z = 1.0 - p * y; return z > 0 ? -2.0 * y * z : 0.0; }
    case NIMFM_LOSS_LOGISTIC: {
      double z = p * y;
      if (z > 0) { double e = exp(-z); return -y * e / (1.0 + e); }
      return -y / (exp(z) + 1.0);
    }
    default: {  // loss.nim:90-93 (sign quirk preserved)
      double z = fabs(y - p);
      return z < thr ? y - p : thr;
    }
  }
}

__host__ __device__ __forceinline__ double loss_mu(int kind) {
  return kind == NIMFM_LOSS_SQUARED_HINGE ? 2.0 : (kind == NIMFM_LOSS_LOGISTIC ? 0.25 : 1.0);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

// sum over aligned sub-groups of G lanes (G power of two <= 32); every lane of the warp must call
__device__ __forceinline__ double group_sum(double v, int G) {
  for (int off = G >> 1; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

// block-wide sum; result valid in thread 0.  red must hold blockDim.x/32 doubles.
__device__ __forceinline__ double block_sum(double v, double *red) {
  v = warp_sum(v);
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  double r = 0.0;
  if (wid == 0) {
    int nw = (blockDim.x + 31) >> 5;
    r = lane < nw ? red[lane] : 0.0;
    r = warp_sum(r);
  }
  return r;
}

// The ANOVA dynamic program / derivative recurrence (sgd.nim:151-170, 176-188) for a RUN-TIME degree M with the state in
// REGISTERS: the loops are unrolled over the compile-time maximum and predicated on M, so A[] is never indexed
// dynamically.  (A dynamically indexed A[] lives in local memory: the sequential solvers' forward pass measured
// 490 cycles per nonzero that way, two thirds of a sample's time.)
typedef double AnovaState[NIMFM_MAX_DEGREE + 1];
__device__ __forceinline__ void anova_init(AnovaState &A) {
  A[0] = 1.0;
#pragma unroll
  for (int t = 1; t <= NIMFM_MAX_DEGREE; ++t) A[t] = 0.0;
}
__device__ __forceinline__ void anova_step(AnovaState &A, int M, double tv) {   // a[t] += a[t-1] * tv, t = M .. 1
#pragma unroll
  for (int t = NIMFM_MAX_DEGREE; t >= 1; --t)
    if (t <= M) A[t] += A[t - 1] * tv;
}
__device__ __forceinline__ double anova_at(const AnovaState &A, int M) {
  double r = A[1];
#pragma unroll
  for (int t = 2; t <= NIMFM_MAX_DEGREE; ++t)
    if (t == M) r = A[t];
  return r;
}
__device__ __forceinline__ double anova_deriv(const AnovaState &A, int M, double x, double p) {   // M != 2
  double g = x;
#pragma unroll
  for (int t = 1; t < NIMFM_MAX_DEGREE; ++t)
    if (t < M) g = x * (A[t] - p * g);
  return g;
}

// The forward DP over a row slice staged in shared memory, col[u * stride] = P[j_u][o][s], for a RUN-TIME degree M
// dispatched ONCE to a compile-time instantiation.  With M tested inside the loop the compiler emits a chain of
// branches per nonzero (measured: 136 cycles per nonzero in the sequential solvers' forward pass, 30 % of a sample);
// the fixed-degree loops are M FP64 operations per nonzero, the loads software-pipelined by the unroll.  Same
// operation order as anova_step / the reference (sgd.nim:151-170); M == 2 keeps its closed form (A[1], A[2] = sums).
template <int M>
__device__ __forceinline__ void anova_forward_fixed(AnovaState &A, const double *col, int stride, const double *X, int z) {
  double a[M + 1];
  a[0] = 1.0;
#pragma unroll
  for (int t = 1; t <= M; ++t) a[t] = 0.0;
#pragma unroll 4
  for (int u = 0; u < z; ++u) {
    const double tv = col[u * stride] * X[u];
    if (M == 2) {
      a[1] += tv;
      a[2] += tv * tv;
    } else {
#pragma unroll
      for (int t = M; t >= 1; --t) a[t] += a[t - 1] * tv;
    }
  }
#pragma unroll
  for (int t = 1; t <= M; ++t) A[t] = a[t];
}
// leaves A[0..M] (others zero) and returns the kernel value of the slot
__device__ __forceinline__ double anova_forward_smem(AnovaState &A, int M, const double *col, int stride, const double *X,
                                                     int z) {
  anova_init(A);
  switch (M) {
    case 1: anova_forward_fixed<1>(A, col, stride, X, z); break;
    case 2: anova_forward_fixed<2>(A, col, stride, X, z); break;
    case 3: anova_forward_fixed<3>(A, col, stride, X, z); break;
    case 4: anova_forward_fixed<4>(A, col, stride, X, z); break;
    case 5: anova_forward_fixed<5>(A, col, stride, X, z); break;
    default: anova_forward_fixed<NIMFM_MAX_DEGREE>(A, col, stride, X, z); break;
  }
  return M == 2 ? (A[1] * A[1] - A[2]) / 2.0 : anova_at(A, M);
}

// element e = tid + r*nth of a row slice [z][SB8] as (u, off) = (e / SB8, e % SB8) WITHOUT a division per element: the
// single-block sequential solvers walk thousands of such elements per sample and a runtime integer division costs
// ~35 instructions.  start() is evaluated once per kernel (tid, nth and SB8 never change), next() is two adds.
struct ElemWalk {
  int u, off, du, doff, SB8;
  __device__ __forceinline__ void start(int tid, int nth, int sb8) {
    SB8 = sb8;
    u = tid / sb8;
    off = tid - u * sb8;
    du = nth / sb8;
    doff = nth - du * sb8;
  }
  __device__ __forceinline__ void next() {
    u += du;
    off += doff;
    if (off >= SB8) {
      off -= SB8;
      ++u;
    }
  }
};

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async8(void *smem, const void *gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

#endif  // __CUDACC__
