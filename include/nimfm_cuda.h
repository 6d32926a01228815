/*
 * nimfm_cuda.h -- C ABI of libnimfm_cuda.so, the B200 (sm_100a) implementation of nimfm's
 * ANOVA-kernel hot path.  Plain pointers and sizes only; no C++/torch types cross this boundary.
 *
 * The reference (neonnnnn/nimfm 0.3.0, pure Nim) has no FFI seam for this path; every entry point
 * below replaces an exported Nim proc (cited as file:line relative to /root/reference/src/nimfm/)
 * and is what nimfm's Nim modules would bind with {.importc, dynlib: "libnimfm_cuda.so".}
 * (binding stubs: nim/nimfm_cuda.nim, INTEGRATION.md).  Mapping: Nim int -> int64_t,
 * float64 -> double, bool -> int32_t, seq[T] -> (const T*, length).
 *
 * Conventions
 *  - every function returns NIMFM_OK (0) or a negative nimfm_status; the message is available from
 *    nimfm_last_error(ctx) (the Nim shim raises ValueError with it, like factorization_machine.nim:114).
 *  - host arrays are COPIED; the caller keeps ownership.  Handles are opaque, owned by the library,
 *    freed explicitly.  One host thread per ctx; calls return after the stream is synchronised unless
 *    the name ends in _async.
 *  - parameter arrays cross the ABI in the REFERENCE layouts: FM P[order][s][j] with j < d+nAug
 *    (factorization_machine.nim:33-36), FFM P[field][j][s] (field_aware_factorization_machine.nim:16-17).
 *    The device layouts (DESIGN.md) are private to the library, as sgd.transpose (sgd.nim:92-96) is
 *    private to the solvers.
 *  - there is NO CPU fallback: without a CUDA device nimfm_ctx_create fails with NIMFM_ERR_CUDA.
 */
#ifndef NIMFM_CUDA_H
#define NIMFM_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  NIMFM_OK = 0,
  NIMFM_ERR_INVALID = -1,   /* bad argument / shape mismatch (reference: ValueError) */
  NIMFM_ERR_CUDA = -2,      /* CUDA runtime error, or no device */
  NIMFM_ERR_NCCL = -3,      /* NCCL error, or communicator not initialised */
  NIMFM_ERR_UNSUPPORTED = -4,
  NIMFM_ERR_STATE = -5      /* call order violated (e.g. solver state not initialised) */
} nimfm_status;

/* loss.nim:15-102 */
typedef enum { NIMFM_LOSS_SQUARED = 0, NIMFM_LOSS_SQUARED_HINGE = 1, NIMFM_LOSS_LOGISTIC = 2, NIMFM_LOSS_HUBER = 3 } nimfm_loss;
/* optimizer/sgd.nim:8-12 SchedulingKind */
typedef enum { NIMFM_SCHED_CONSTANT = 0, NIMFM_SCHED_OPTIMAL = 1, NIMFM_SCHED_INVSCALING = 2, NIMFM_SCHED_PEGASOS = 3 } nimfm_sched;
/* prox for MBPSGD (minibatch_psgd.nim:119-121): identity == any regulariser at gamma=0; L1 == l1.nim:38-41;
 * SQUAREDL12 == newSquaredL12(transpose=true), the MBPSGD default (squaredl12.nim:147-156: one vector per
 * component over all features; degree 2 only, :103-106); SQUAREDL12_ROWS == transpose=false (:157-159);
 * L21 == l21.nim:25-35 */
typedef enum {
  NIMFM_REG_IDENTITY = 0, NIMFM_REG_L1 = 1, NIMFM_REG_SQUAREDL12 = 2, NIMFM_REG_SQUAREDL12_ROWS = 3, NIMFM_REG_L21 = 4
} nimfm_reg;
typedef enum { NIMFM_DS_CSR = 0, NIMFM_DS_CSC = 1, NIMFM_DS_CSR_FIELD = 2 } nimfm_ds_kind;

typedef struct nimfm_ctx nimfm_ctx;
typedef struct nimfm_dataset nimfm_dataset;
typedef struct nimfm_fm nimfm_fm;
typedef struct nimfm_ffm nimfm_ffm;

/* ---------------------------------------------------------------- lifecycle */
int32_t nimfm_ctx_create(int32_t device, nimfm_ctx **out);
int32_t nimfm_ctx_destroy(nimfm_ctx *ctx);
const char *nimfm_last_error(const nimfm_ctx *ctx);
/* library/ABI version (major*100 + minor) and the number of kernels launched by this ctx so far */
int32_t nimfm_version(void);
int64_t nimfm_launch_count(const nimfm_ctx *ctx);
/* what the last host-fed call (nimfm_fm_loss_grad_host / nimfm_fm_decision_function_host) moved over the link:
 * bytes host->device, bytes device->host, and the host staging threads it used (0: ids narrowed on the device) */
/* free / total bytes of the context's device (cudaMemGetInfo) */
int32_t nimfm_mem_info(nimfm_ctx *ctx, int64_t *freeBytes, int64_t *totalBytes);
int32_t nimfm_stream_stats(const nimfm_ctx *ctx, int64_t *h2dBytes, int64_t *d2hBytes, int32_t *hostThreads);
/* Page-lock / release a caller-owned host array (cudaHostRegister) for as long as its owner -- the dataset object
 * holding the seqs of tensor/sparse.nim:4-31 -- lives: the host-fed calls then copy straight out of it at link
 * rate.  Unregistered (pageable) arrays still work: the host staging team copies them through pinned slots. */
int32_t nimfm_host_register(nimfm_ctx *ctx, const void *ptr, int64_t bytes);
int32_t nimfm_host_unregister(nimfm_ctx *ctx, const void *ptr);

/* Multi-GPU (one process per GPU).  The reference has no distributed backend (SURVEY 2a); this is
 * the synchronous data-parallel replacement of its Hogwild threads (sgd_multi.nim:86-95).
 * uid is NCCL_UNIQUE_ID_BYTES (128) bytes obtained on rank 0 and broadcast by the host. */
int32_t nimfm_comm_unique_id(void *uid128);
int32_t nimfm_comm_init(nimfm_ctx *ctx, int32_t rank, int32_t nranks, const void *uid128);
int32_t nimfm_comm_size(const nimfm_ctx *ctx);
/* `count` int64 values of every rank, rank-major (all[r*count + i]), on every host: what the host side needs to
 * agree on before a sharded fit() -- global nSamples / nnz behind MBPSGD's default minibatch
 * (minibatch_psgd.nim:157-165), shard lengths.  One rank: a copy.  count <= 4096. */
int32_t nimfm_comm_allgather_i64(nimfm_ctx *ctx, const int64_t *mine, int32_t count, int64_t *all);

/* ---------------------------------------------------------------- datasets
 * newCSRDataset / newCSCDataset / newCSRFieldDataset (dataset.nim:116-153).  indices are narrowed to
 * int32 on the device when d (resp. n) < 2^31.  [rowBegin,rowEnd) uploads a row shard of a CSR
 * (== X[slice], tensor/sparse.nim:263-290) with indptr rebased; pass 0,n for everything. */
int32_t nimfm_csr_upload(nimfm_ctx *ctx, int64_t n, int64_t d, const double *data,
                         const int64_t *indices, const int64_t *indptr, const int64_t *fields,
                         int64_t nFields, int64_t rowBegin, int64_t rowEnd, nimfm_dataset **out);
int32_t nimfm_csc_upload(nimfm_ctx *ctx, int64_t n, int64_t d, const double *data,
                         const int64_t *indices, const int64_t *indptr, nimfm_dataset **out);
/* toCSCDataset / toCSRDataset (dataset.nim:418-427 -> tensor/sparse.nim:490-527): stable counting sort,
 * run on the device as a stable radix sort by the other axis (bit-exact: same indptr, same order) */
int32_t nimfm_dataset_transpose(nimfm_ctx *ctx, const nimfm_dataset *in, nimfm_dataset **out);
/* X[indicesRow] for CSRDataset / CSRFieldDataset (dataset.nim:319-367 -> tensor/sparse.nim:263-285).
 * Targets set on `in` are gathered too (== shuffle(X, y, indices), dataset.nim:372-381).  Out-of-range
 * ids fail with the reference's messages (sparse.nim:254-260). */
int32_t nimfm_dataset_take_rows(nimfm_ctx *ctx, const nimfm_dataset *in, const int64_t *rowIdx,
                                int64_t nIdx, nimfm_dataset **out);
/* X[first..last], INCLUSIVE like Nim's Slice (dataset.nim:328-348): CSR kinds gather the rows; a CSC
 * is filtered per column in O(nnz) with row ids rebased (tensor/sparse.nim:300-325). */
int32_t nimfm_dataset_slice_rows(nimfm_ctx *ctx, const nimfm_dataset *in, int64_t first, int64_t last,
                                 nimfm_dataset **out);
/* vstack (dataset.nim:452-483 -> tensor/sparse.nim:564-640): all parts of one kind and nFeatures */
int32_t nimfm_dataset_vstack(nimfm_ctx *ctx, const nimfm_dataset *const *parts, int32_t nParts,
                             nimfm_dataset **out);
/* targets of fit(X, y, fm); length = nSamples of the (shard of the) dataset */
int32_t nimfm_dataset_set_targets(nimfm_ctx *ctx, nimfm_dataset *ds, const double *y);
int32_t nimfm_dataset_info(const nimfm_dataset *ds, int64_t *n, int64_t *d, int64_t *nnz,
                           int32_t *kind, int64_t *nFields, int64_t *maxRowNnz);
/* read the device arrays back in the reference dtypes (bit-exact bookkeeping checks) */
int32_t nimfm_dataset_download(nimfm_ctx *ctx, const nimfm_dataset *ds, double *data,
                               int64_t *indices, int64_t *indptr, int64_t *fields);
int32_t nimfm_dataset_free(nimfm_ctx *ctx, nimfm_dataset *ds);
/* Text loaders (parsed by all host cores, uploaded straight to the device; targets are set on the
 * dataset and read back with nimfm_dataset_get_targets).  nFeatures / nFields <= 0: inferred.
 * loadSVMLightFile (dataset.nim:562-693; asCsc != 0 gives the CSCDataset overload, :643-686),
 * loadFFMFile (dataset.nim:696-790), loadUserItemRatingFile (dataset.nim:840-990). */
int32_t nimfm_load_svmlight(nimfm_ctx *ctx, const char *path, int64_t nFeatures, int32_t asCsc,
                            nimfm_dataset **out);
int32_t nimfm_load_ffm(nimfm_ctx *ctx, const char *path, int64_t nFeatures, int64_t nFields,
                       nimfm_dataset **out);
int32_t nimfm_load_user_item_rating(nimfm_ctx *ctx, const char *path, int32_t asCsc, nimfm_dataset **out);
/* STREAMCSR / STREAMCSC binary files (tensor/sparse_stream.nim:3-33; written by convertSVMLightFile /
 * transposeFile, dataset.nim:1017-1200) loaded WHOLE into a device CSR / CSC dataset (newStreamCSRDataset /
 * newStreamCSCDataset, dataset.nim:170-179, without the window cache); pathY (nullable) is the raw float64
 * label file of loadStreamLabel (dataset.nim:995-1014). */
int32_t nimfm_load_stream(nimfm_ctx *ctx, const char *pathX, const char *pathY, nimfm_dataset **out);
/* The window cache (tensor/sparse_stream.nim:232-270; StreamCSRDataset, dataset.nim:1017-1402) with HBM as the
 * cache: an open handle indexes the file's segments once, nimfm_stream_window_end sizes a window of at most
 * maxBytes of file payload (>= 1 row), nimfm_stream_load_window makes rows [segBegin, segEnd) a resident CSR
 * dataset (indptr rebased, labels attached when pathY was given).  A file larger than device memory is
 * processed window by window; StreamCSC files load whole only (a window of columns is another matrix). */
typedef struct nimfm_stream nimfm_stream;
int32_t nimfm_stream_open(nimfm_ctx *ctx, const char *pathX, const char *pathY, nimfm_stream **out);
int32_t nimfm_stream_info(const nimfm_stream *sh, int32_t *kind, int64_t *nRows, int64_t *nCols, int64_t *nnz,
                          int64_t *maxSegNnz, int64_t *payloadBytes);
int64_t nimfm_stream_window_end(const nimfm_stream *sh, int64_t segBegin, int64_t maxBytes);
int32_t nimfm_stream_load_window(nimfm_ctx *ctx, nimfm_stream *sh, int64_t segBegin, int64_t segEnd,
                                 nimfm_dataset **out);
int32_t nimfm_stream_close(nimfm_stream *sh);
int32_t nimfm_dataset_get_targets(nimfm_ctx *ctx, const nimfm_dataset *ds, double *y);

/* ---------------------------------------------------------------- FM model state
 * FactorizationMachine (model/factorization_machine.nim:11-139).  nOrders / nAug follow :81-97.
 * 1 <= degree <= 6.  nOrders = 0 if and only if degree = 1: the linear model b + <w, x>, which has no P (nAugments
 * must be 0 as well).  Every array argument shaped like P (P, gP, the AdaGrad gsP / gnP) may be NULL when the
 * model has no P, and nothing is copied for it. */
int32_t nimfm_fm_create(nimfm_ctx *ctx, int32_t degree, int32_t nComponents, int32_t nOrders,
                        int32_t nAugments, int64_t nFeatures, int32_t fitLinear,
                        int32_t fitIntercept, nimfm_fm **out);
int32_t nimfm_fm_set_params(nimfm_ctx *ctx, nimfm_fm *fm, const double *P, const double *w,
                            double intercept, const double *lams /* NULL == ones */);
int32_t nimfm_fm_get_params(nimfm_ctx *ctx, nimfm_fm *fm, double *P, double *w, double *intercept);
int32_t nimfm_fm_free(nimfm_ctx *ctx, nimfm_fm *fm);

/* decisionFunction (model/factorization_machine.nim:100-122; kernels.nim:4-64): out[n] on the host.
 * Accepts a CSR (row kernel) or a CSC dataset (column kernel). */
int32_t nimfm_fm_decision_function(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, double *out);

/* predict + gradient of one minibatch: predictWithGrad (optimizer/sgd.nim:191-202) followed by
 * updateGradient's scatter (optimizer/minibatch_psgd.nim:67-88) for rows
 *   rowIdx[0..nRows)            if rowIdx != NULL, else
 *   (rowBegin + q) mod n, q<nRows
 * with coef = dloss / miniBatchSize.  Gradients accumulate into the model's device gradient buffers
 * (zeroed first when zeroGrads != 0; all-reduced over the communicator when allreduce != 0).
 * lossSum (nullable) receives the sum of loss values of the rows processed on THIS rank. */
int32_t nimfm_fm_loss_grad(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, int32_t loss,
                           double huberThreshold, int64_t rowBegin, int64_t nRows,
                           const int64_t *rowIdx, int64_t miniBatchSize, int32_t zeroGrads,
                           int32_t allreduce, double *lossSum);
/* The same predict+grad step fed from HOST buffers (the end-to-end path): rows [0,nRows) of a host
 * CSR in the reference dtypes (f64 data, i64 indices / indptr, f64 y) are streamed to the device in
 * chunks of chunkRows rows (<=0: library default), the host->device copy of chunk c+1 overlapping
 * the kernel of chunk c on a second stream; ids are narrowed to int32 and indptr rebased by the library's
 * host staging threads (or on the device when a rank has too few host threads to itself).  Page-locked
 * arrays (nimfm_host_register, cudaHostAlloc) are read by the copy engine directly; PAGEABLE arrays -- a Nim
 * seq -- are detected (cudaPointerGetAttributes) and their values / targets go through the same staging
 * threads into pinned slots, so no copy is left to the driver's single-threaded pageable path. */
int32_t nimfm_fm_loss_grad_host(nimfm_ctx *ctx, nimfm_fm *fm, int64_t nRows, int64_t d, const double *data,
                                const int64_t *indices, const int64_t *indptr, const double *y,
                                int32_t loss, double huberThreshold, int64_t miniBatchSize,
                                int64_t chunkRows, int32_t zeroGrads, int32_t allreduce, double *lossSum);
/* decisionFunction fed from HOST buffers the same way (out[nRows] on the host): the serving-side call */
int32_t nimfm_fm_decision_function_host(nimfm_ctx *ctx, nimfm_fm *fm, int64_t nRows, int64_t d,
                                        const double *data, const int64_t *indices, const int64_t *indptr,
                                        int64_t chunkRows, double *out);
/* read the gradient buffers back in the reference layout (gP[order][s][j], gw[d], gb) */
int32_t nimfm_fm_get_grads(nimfm_ctx *ctx, nimfm_fm *fm, double *gP, double *gw, double *gb);

/* ---------------------------------------------------------------- MBPSGD (optimizer/minibatch_psgd.nim) */
typedef struct {
  int32_t loss;            /* nimfm_loss */
  double huberThreshold;
  double eta0, alpha0, alpha, beta, gamma;      /* newMBPSGD, :25-30 */
  int32_t reg;             /* nimfm_reg */
  int32_t scheduling;      /* nimfm_sched */
  double power;
  int64_t miniBatchSize;   /* resolved by the host as in :157-165 (must be >= 1) */
  int64_t maxIterInner;    /* resolved by the host (must be >= 1) */
} nimfm_mbpsgd_cfg;
/* One epoch() (:91-124).  *it is MBPSGD.it (in/out), *ii the sample cursor (in/out).  sampleIdx is
 * NULL for cyclic order from *ii (shuffle=false) or the miniBatchSize*maxIterInner row ids the
 * host's cursor+shuffle logic (:102-111) yields for this epoch.  With a communicator every rank
 * passes its own shard (miniBatchSize is the GLOBAL size used in coef; each rank processes localBatch
 * rows per inner iteration; the shares may differ but must add up to miniBatchSize, and miniBatchSize,
 * maxIterInner and *it must agree across ranks -- checked).  Per minibatch the gradient pool is
 * reduce-scattered, every rank runs Params.step (params.nim:90-98) and the prox on its 1/N slice of
 * [P | w | b], and the parameters are all-gathered (the column-wise SquaredL12 prox, which sums over all
 * features, keeps an all-reduce followed by the identical dense step on every rank). */
int32_t nimfm_fm_mbpsgd_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X,
                              const nimfm_mbpsgd_cfg *cfg, int64_t localBatch, int64_t *it,
                              int64_t *ii, const int64_t *sampleIdx, double *runningLoss);

/* ---------------------------------------------------------------- AdaGrad (optimizer/adagrad.nim) */
typedef struct {
  int32_t loss;
  double huberThreshold;
  double eta0, alpha0, alpha, beta, eps;        /* newAdaGrad, :20-22 */
  int64_t miniBatchSize;   /* 1 == the reference's per-sample semantics; >1 == synchronous minibatch */
} nimfm_adagrad_cfg;
/* AdaGrad.init (:47-62): allocate g_sum / g_norm, g_sum=0, g_norm=eps (only when reset != 0) */
int32_t nimfm_fm_adagrad_init(nimfm_ctx *ctx, nimfm_fm *fm, double eps, int32_t reset);
/* one pass over perm[0..nRows) (NULL == 0..n-1) in batches of cfg->miniBatchSize (:164-181);
 * *it in/out; viol / lossSum are the epoch sums (:172-176). */
int32_t nimfm_fm_adagrad_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X,
                               const nimfm_adagrad_cfg *cfg, int64_t *it, const int64_t *perm,
                               int64_t nRows, double *viol, double *lossSum);
/* AdaGrad.finalize (:65-84): closed form over ALL parameters with t = it-1 */
int32_t nimfm_fm_adagrad_finalize(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_adagrad_cfg *cfg, int64_t it);
/* optimizer state for warm starts (AdaGrad.g_sum / g_norm, :15-16), SOLVER layout [order][j][s] */
int32_t nimfm_fm_adagrad_get_state(nimfm_ctx *ctx, nimfm_fm *fm, double *gsP, double *gnP, double *gsw,
                                   double *gnw, double *gsb, double *gnb);
int32_t nimfm_fm_adagrad_set_state(nimfm_ctx *ctx, nimfm_fm *fm, const double *gsP, const double *gnP,
                                   const double *gsw, const double *gnw, double gsb, double gnb);

/* ---------------------------------------------------------------- SGD (optimizer/sgd.nim) */
typedef struct {
  int32_t loss;
  double huberThreshold;
  double eta0, alpha0, alpha, beta;             /* newSGD, :23-25 */
  int32_t scheduling;
  double power;
} nimfm_sgd_cfg;
/* SGD is sequential per sample (each step reads the parameters the previous one wrote, :246-258),
 * so the device runs the sample loop inside ONE persistent thread block: exact reference semantics,
 * "replicas only" for multi-GPU.  begin resets the lazy-scaling caches (:269-272); epoch runs
 * step() over perm (:296-300); end applies finalize (:99-113). */
int32_t nimfm_fm_sgd_begin(nimfm_ctx *ctx, nimfm_fm *fm);
int32_t nimfm_fm_sgd_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_sgd_cfg *cfg,
                           int64_t *it, const int64_t *perm, int64_t nRows, double *viol, double *lossSum);
int32_t nimfm_fm_sgd_end(nimfm_ctx *ctx, nimfm_fm *fm);

/* ---------------------------------------------------------------- PSGD (optimizer/psgd.nim) */
typedef struct {
  int32_t loss;
  double huberThreshold;
  double eta0, alpha0, alpha, beta, gamma;      /* newPSGD, psgd.nim:22-25 */
  int32_t reg;             /* NIMFM_REG_L1 | _L21 (lazy protocols, l1.nim:84-136 / l21.nim:36-112) |
                              _SQUAREDL12 | _SQUAREDL12_ROWS (dense step + full prox, squaredl12.nim:199-230) */
  int32_t scheduling;
  double power;
} nimfm_psgd_cfg;
/* Sequential per sample like SGD ("replicas only").  begin == reg.initSGD + the scaling caches
 * (psgd.nim:98-112); epoch == the sample loop over perm (NULL: 0..nRows-1) (:118-176), lossSum its loss
 * sum; end == finalize (:58-75). */
int32_t nimfm_fm_psgd_begin(nimfm_ctx *ctx, nimfm_fm *fm);
int32_t nimfm_fm_psgd_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_psgd_cfg *cfg,
                            int64_t *it, const int64_t *perm, int64_t nRows, double *lossSum);
int32_t nimfm_fm_psgd_end(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_psgd_cfg *cfg);

/* ---------------------------------------------------------------- CD (optimizer/cd.nim) */
typedef struct {
  int32_t loss;
  double huberThreshold;
  double alpha0, alpha, beta;                   /* newCD (:12-13), NOT yet multiplied by nSamples */
} nimfm_cd_cfg;
/* begin == the cache set-up of fit (:123-151): scaled alphas, colNormSq, yPred; X must be CSC with targets.
 * epoch == one outer iteration (:156-172): intercept, linear, then epoch/epochDeg2 per order;
 * returns viol, the mean loss (:177-181) and regularization/n (:182-183). */
int32_t nimfm_fm_cd_begin(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *Xcsc, const nimfm_cd_cfg *cfg);
int32_t nimfm_fm_cd_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *Xcsc, const nimfm_cd_cfg *cfg,
                          double *viol, double *lossMean, double *regOverN);
/* PCD (optimizer/pcd.nim:38-200): cd.fit's sweeps with the sparsity regulariser's per-coordinate prox
 * (L1: l1.nim:22-24; SquaredL12, either orientation: squaredl12.nim:108-114,161-185) and the
 * invStepSize guard in every sweep (:55,96).  Uses nimfm_fm_cd_begin / _end / _get_ypred.
 * regOverN is regularization/n without the gamma*reg.eval term (:181-183, printed by the host). */
typedef struct {
  int32_t loss;
  double huberThreshold;
  double alpha0, alpha, beta, gamma;            /* newPCD (:17-20), NOT yet multiplied by nSamples */
  int32_t reg;                                  /* NIMFM_REG_L1 | NIMFM_REG_SQUAREDL12 | NIMFM_REG_SQUAREDL12_ROWS */
} nimfm_pcd_cfg;
int32_t nimfm_fm_pcd_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *Xcsc, const nimfm_pcd_cfg *cfg,
                           double *viol, double *lossMean, double *regOverN);
int32_t nimfm_fm_cd_get_ypred(nimfm_ctx *ctx, nimfm_fm *fm, double *yPred);
int32_t nimfm_fm_cd_end(nimfm_ctx *ctx, nimfm_fm *fm);

/* ---------------------------------------------------------------- FFM
 * FieldAwareFactorizationMachine (model/field_aware_factorization_machine.nim:6-92) */
int32_t nimfm_ffm_create(nimfm_ctx *ctx, int32_t nComponents, int64_t nFields, int64_t nFeatures,
                         int32_t fitLinear, int32_t fitIntercept, nimfm_ffm **out);
int32_t nimfm_ffm_set_params(nimfm_ctx *ctx, nimfm_ffm *m, const double *P, const double *w, double intercept);
int32_t nimfm_ffm_get_params(nimfm_ctx *ctx, nimfm_ffm *m, double *P, double *w, double *intercept);
int32_t nimfm_ffm_free(nimfm_ctx *ctx, nimfm_ffm *m);
/* decisionFunction (:52-76) */
int32_t nimfm_ffm_decision_function(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, double *out);
/* predictWithGrad (optimizer/sgd_ffm.nim:11-30) + minibatch-mean gradient scatter, as nimfm_fm_loss_grad */
int32_t nimfm_ffm_loss_grad(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, int32_t loss,
                            double huberThreshold, int64_t rowBegin, int64_t nRows, const int64_t *rowIdx,
                            int64_t miniBatchSize, int32_t zeroGrads, int32_t allreduce, double *lossSum);
int32_t nimfm_ffm_get_grads(nimfm_ctx *ctx, nimfm_ffm *m, double *gP, double *gw, double *gb);
/* AdaGrad for FFM (optimizer/adagrad_ffm.nim:11-66 over adagrad.nim:87-134 with order == field) */
int32_t nimfm_ffm_adagrad_init(nimfm_ctx *ctx, nimfm_ffm *m, double eps, int32_t reset);
int32_t nimfm_ffm_adagrad_epoch(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X,
                                const nimfm_adagrad_cfg *cfg, int64_t *it, const int64_t *perm,
                                int64_t nRows, double *viol, double *lossSum);
int32_t nimfm_ffm_adagrad_finalize(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_adagrad_cfg *cfg, int64_t it);
/* optimizer state for warm starts (AdaGrad.g_sum / g_norm, adagrad.nim:15-16, kept by init when warmStart and the
 * shapes match, :47-62), gsP / gnP in the REFERENCE layout [field][j][s] of ffm.P.  Both need nimfm_ffm_adagrad_init
 * first (else NIMFM_ERR_STATE); set_state takes no NULL array. */
int32_t nimfm_ffm_adagrad_get_state(nimfm_ctx *ctx, nimfm_ffm *m, double *gsP, double *gnP, double *gsw,
                                    double *gnw, double *gsb, double *gnb);
int32_t nimfm_ffm_adagrad_set_state(nimfm_ctx *ctx, nimfm_ffm *m, const double *gsP, const double *gnP,
                                    const double *gsw, const double *gnw, double gsb, double gnb);
/* Synchronous-minibatch SGD: the deterministic device analogue of the Hogwild variants fit(..., maxThreads)
 * (optimizer/sgd_multi.nim:40-120, sgd_ffm_multi.nim:31-103).  The miniBatchSize samples of a minibatch are
 * evaluated at the same parameters and their updates applied at once with the step sizes of the minibatch's
 * first iteration: touched features p <- (1-eta beta)^B p - eta sum_i dL_i dA_i (viol += |p_new - p|),
 * untouched features p <- (1-eta beta)^B p, it += B.  miniBatchSize = 1 is step() itself (sgd.nim:205-258).
 * No begin / end: the parameters stay canonical between calls.  perm (nullable): sample order.
 * Data parallel like nimfm_fm_mbpsgd_epoch: with a communicator X is this rank's shard, localBatch (<= 0: =
 * miniBatchSize) the rows this rank feeds per minibatch, miniBatchSize = localBatch x ranks the global one;
 * touch counts and gradients are all-reduced, every rank applies the identical step.  Shards and shares may be
 * uneven: every rank runs max_r ceil(nRows_r / localBatch_r) minibatches (feeding 0 rows once its shard is used
 * up) and `it` advances by the global row count of each minibatch; the same holds for the AdaGrad epochs. */
int32_t nimfm_fm_sgd_minibatch_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_sgd_cfg *cfg,
                                     int64_t miniBatchSize, int64_t localBatch, int64_t *it, const int64_t *perm,
                                     int64_t nRows, double *viol, double *lossSum);
int32_t nimfm_ffm_sgd_minibatch_epoch(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X,
                                      const nimfm_sgd_cfg *cfg, int64_t miniBatchSize, int64_t localBatch,
                                      int64_t *it, const int64_t *perm, int64_t nRows, double *viol,
                                      double *lossSum);
/* SGD for FFM (optimizer/sgd_ffm.nim:33-106), sequential like nimfm_fm_sgd_* */
int32_t nimfm_ffm_sgd_begin(nimfm_ctx *ctx, nimfm_ffm *m);
int32_t nimfm_ffm_sgd_epoch(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, const nimfm_sgd_cfg *cfg,
                            int64_t *it, const int64_t *perm, int64_t nRows, double *viol, double *lossSum);
int32_t nimfm_ffm_sgd_end(nimfm_ctx *ctx, nimfm_ffm *m);

/* ---------------------------------------------------------------- measurement hooks (bench.py)
 * Run `reps` back-to-back launches of the named hot-path kernel on device-resident data and return
 * the average device time per launch in milliseconds (CUDA events on the library's stream). */
int32_t nimfm_fm_time_loss_grad(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, int32_t loss,
                                int64_t nRows, int64_t miniBatchSize, int32_t reps, int32_t gradToo,
                                float *msPerLaunch);
int32_t nimfm_ffm_time_loss_grad(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, int32_t loss,
                                 int64_t nRows, int64_t miniBatchSize, int32_t reps, int32_t gradToo,
                                 float *msPerLaunch);
/* device-time stopwatch on the library's stream (CUDA events): start, run any calls, stop -> ms */
int32_t nimfm_timer_start(nimfm_ctx *ctx);
int32_t nimfm_timer_stop(nimfm_ctx *ctx, float *ms);
/* raw device pointers of the gradient buffers (so a host that prefers its own collective, e.g.
 * torch.distributed, can all-reduce them in place): P part then w part then [gb, lossSum] */
int32_t nimfm_fm_grad_device_ptr(nimfm_fm *fm, void **ptr, int64_t *nDoubles);

#ifdef __cplusplus
}
#endif
#endif /* NIMFM_CUDA_H */
