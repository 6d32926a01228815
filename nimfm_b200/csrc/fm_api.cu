// fm_api.cu -- FactorizationMachine state on the device and the row-parallel entry points:
// decisionFunction (K1), predict+grad (K2), MBPSGD epoch (K2+K3), AdaGrad epoch (K4+K5).
#include <math.h>

#include <stdlib.h>

#include <algorithm>
#include <memory>

#include "dense_kernels.cuh"
#include "fm_rows_stream.cuh"
#include "prox_kernels.cuh"
#include "adagrad_seq.cuh"
#include "host_stage.h"

// ------------------------------------------------------------------ layout permutations
// reference model layout  R[o][s][j]   (factorization_machine.nim:33-36)
// reference solver layout S[o][j][s]   (sgd.nim:92-96)
// device layout           D[j][o][s]
__global__ void permute_model_to_dev(const double *R, double *D, int nO, int k, int64_t dd) {
  const int64_t total = (int64_t)nO * k * dd;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(e % k);
    const int64_t t = e / k;
    const int o = (int)(t % nO);
    const int64_t j = t / nO;
    D[e] = R[((int64_t)o * k + s) * dd + j];
  }
}
__global__ void permute_dev_to_model(const double *D, double *R, int nO, int k, int64_t dd) {
  const int64_t total = (int64_t)nO * k * dd;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = e % dd;
    const int64_t t = e / dd;
    const int s = (int)(t % k);
    const int o = (int)(t / k);
    R[e] = D[(j * nO + o) * k + s];
  }
}
__global__ void permute_solver_dev(const double *S, double *D, int nO, int k, int64_t dd, int toDev) {
  const int64_t total = (int64_t)nO * k * dd;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(e % k);
    const int64_t t = e / k;
    const int o = (int)(t % nO);
    const int64_t j = t / nO;
    const int64_t se = ((int64_t)o * dd + j) * k + s;
    if (toDev) D[e] = S[se];
    else const_cast<double *>(S)[se] = D[e];
  }
}

// ------------------------------------------------------------------ launch planning
int nimfm_fm_det_loss_grad(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const RowPlan &pl, int loss, double thr,
                           int64_t rowBegin, int64_t nRows, double mb, double *yOutDev, const RowArgs &base);
int nimfm_fm_det_pass(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_det_twin *tw, const RowPlan &pl, int loss, double thr,
                      int64_t rowBegin, int64_t nRows, double mb, double *yOutDev, const RowArgs &base,
                      const FmDetTargets &o);

static bool is_explicit(const nimfm_fm *fm) { return fm->degree > 2 && fm->nOrders == fm->degree - 1; }

// the multiple a rank's flat slice of [P | w | b] is rounded up to: whole (feature, order-block) vectors, an even
// number of doubles; 2 for the linear model (no P)
static int64_t slice_align(const nimfm_fm *fm) {
  const int64_t SB8 = (int64_t)fm->nOrders * fm->k;
  return SB8 == 0 ? 2 : ((SB8 & 1) ? 2 * SB8 : SB8);
}

// Chooses the kernel (the streaming instance when one exists for the shape and no row, dummy features
// included, holds more than 512 nonzeros, else the generic one), the staging capacity CH, the block size
// that maximises resident warps under the shared-memory budget, and a persistent grid of occupancy x
// numSMs blocks.
static int plan_rows(nimfm_ctx *ctx, const nimfm_fm *fm, const nimfm_dataset *X, int64_t nRows, int mode,
                     RowPlan *pl) {
  if (fm->nOrders == 0) return nimfm_fm_linear_plan(ctx, X, nRows, mode, pl);   // degree 1 (fm_linear.cu)
  const int nAcc = (mode == MODE_PREDICT || mode == MODE_STASH) ? 0 : (mode == MODE_GRAD ? 1 : 2);
  const int nHotTot = nAcc ? (X->hotSlot ? X->nHot : 0) + fm->nAug : 0;
  const int k = fm->k;
  const int G = k <= 8 ? 8 : (k <= 16 ? 16 : 32);
  const int gpw = 32 / G;
  const int SB8 = fm->nOrders * k;
  int64_t z = X->maxSegNnz + fm->nAug;
  if (z < 1) z = 1;
  const size_t capPerGroup = 40 * 1024;
  const bool expl = is_explicit(fm);
  RowKernels ks;
  switch (mode) {
    case MODE_PREDICT: ks = row_kernels<MODE_PREDICT>(fm->degree, expl, k); break;
    case MODE_GRAD: ks = row_kernels<MODE_GRAD>(fm->degree, expl, k); break;
    case MODE_ADAGRAD: ks = row_kernels<MODE_ADAGRAD>(fm->degree, expl, k); break;
    default: ks = row_kernels<MODE_STASH>(fm->degree, expl, k); break;
  }
  // NIMFM_ROW_KERNEL=generic forces the generic kernel onto the streaming instance's shapes (and with the generic
  // stash forward, the generic column kernel of the deterministic route)
  const char *env = getenv("NIMFM_ROW_KERNEL");
  const bool stream = ks.stream && z <= 512 && !(env && !strcmp(env, "generic"));
  RowKernel kern = stream ? ks.stream : ks.generic;
  int64_t CH = z;
  size_t perGroup;
  if (stream) {
    perGroup = stream_group_smem((int)CH, SB8, nHotTot, nAcc);
  } else {
    const size_t perNnz = (size_t)SB8 * 8 + 13;
    CH = std::min<int64_t>(z, (int64_t)(capPerGroup / perNnz));
    if (CH < 1)
      return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "nOrders*nComponents=%d too large for the device row kernel", SB8);
    perGroup = row_group_smem((int)CH, SB8, nHotTot, nAcc ? nAcc : 1);
  }
  if (!kern) return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "no row kernel for degree %d", fm->degree);
  int bestBlock = 0, bestOcc = 0, bestWarps = -1;
  cudaFuncAttributes fattr;
  CK(cudaFuncGetAttributes(&fattr, kern));
  for (int block : {256, 128, 64, 32}) {
    const size_t smem = (size_t)(block / 32) * gpw * perGroup;
    if (smem > (size_t)ctx->smemOptin || block > fattr.maxThreadsPerBlock) continue;
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, block, smem));
    const int warps = occ * block / 32;
    if (warps > bestWarps) {
      bestWarps = warps;
      bestBlock = block;
      bestOcc = occ;
    }
  }
  if (bestBlock == 0 || bestOcc == 0)
    return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "row kernel does not fit on an SM (perGroup=%zu B)", perGroup);
  pl->kern = kern;
  pl->stream = stream;
  pl->G = G;
  pl->CH = (int)CH;
  pl->block = bestBlock;
  pl->smem = (size_t)(bestBlock / 32) * gpw * perGroup;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl->smem));
  const int64_t tiles = (nRows + gpw - 1) / gpw;
  const int warpsPerBlock = bestBlock / 32;
  int64_t grid = (tiles + warpsPerBlock - 1) / warpsPerBlock;
  const int64_t cap = (int64_t)bestOcc * ctx->numSMs;
  if (grid > cap) grid = cap;
  if (grid < 1) grid = 1;
  pl->grid = (int)grid;
  pl->nWarps = grid * warpsPerBlock;
  return NIMFM_OK;
}

static int check_fm_ds(nimfm_ctx *ctx, const nimfm_fm *fm, const nimfm_dataset *X, bool needY) {
  REQUIRE(fm && X, "NULL handle");
  REQUIRE(X->kind == NIMFM_DS_CSR || X->kind == NIMFM_DS_CSR_FIELD, "a CSR dataset is required");
  REQUIRE(X->d == fm->d, "Invalid nFeatures. (dataset %lld, model %lld)", (long long)X->d, (long long)fm->d);
  REQUIRE(!needY || X->y != nullptr, "dataset has no targets (nimfm_dataset_set_targets)");
  return NIMFM_OK;
}

static void fill_row_args(RowArgs &a, const nimfm_fm *fm, const nimfm_dataset *X) {
  memset(&a, 0, sizeof(a));
  a.data = X->data;
  a.indices = X->indices;
  a.indptr = X->indptr;
  a.y = X->y;
  a.n = X->n;
  a.k = fm->k;
  a.nAug = fm->nAug;
  a.d = fm->d;
  a.P = fm->P;
  a.w = fm->w;
  a.b = fm->b;
  a.lams = fm->lamsAreOnes ? nullptr : fm->lams;
  a.fitLinear = fm->fitLinear;
  a.fitIntercept = fm->fitIntercept;
  a.mb = 1.0;
  a.hotSlot = X->hotSlot;
  a.hotList = X->hotList;
  a.nHot = X->hotSlot ? X->nHot : 0;
}

extern "C" {

// ================================================================== model state
int32_t nimfm_fm_create(nimfm_ctx *ctx, int32_t degree, int32_t nComponents, int32_t nOrders,
                        int32_t nAugments, int64_t nFeatures, int32_t fitLinear, int32_t fitIntercept,
                        nimfm_fm **out) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(out != nullptr, "out is NULL");
  REQUIRE(degree >= 1, "degree < 1.");
  if (degree > NIMFM_MAX_DEGREE)
    return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "degree %d > %d not instantiated", degree, NIMFM_MAX_DEGREE);
  REQUIRE(nComponents >= 1, "nComponents < 1.");
  if (degree == 1) {   // the linear model: no ANOVA term, no P (factorization_machine.nim:89-97)
    REQUIRE(nOrders == 0, "degree 1 has nOrders = 0 (got %d)", nOrders);
    REQUIRE(nAugments == 0, "degree 1 has no dummy features: nAugments = %d (fitLower = augment with fitLinear gives "
            "degree - 2 = -1 at degree 1)", nAugments);
  } else {
    REQUIRE(nOrders == 1 || nOrders == degree - 1, "nOrders must be 1 or degree-1 (factorization_machine.nim:89-97)");
    REQUIRE(nAugments >= 0 && nAugments < degree, "bad nAugments");
  }
  REQUIRE(nFeatures >= 1, "nFeatures < 1");
  CK(cudaSetDevice(ctx->device));
  nimfm_fm *fm = new nimfm_fm();
  fm->degree = degree;
  fm->k = nComponents;
  fm->nOrders = nOrders;
  fm->nAug = nAugments;
  fm->d = nFeatures;
  fm->fitLinear = fitLinear != 0;
  fm->fitIntercept = fitIntercept != 0;
  const int64_t nP = fm->nP(), d = fm->d;
  // slack: room to round a rank's flat slice up to whole (feature, order-block) vectors for up to 64 ranks
  fm->poolCap = nP + d + 8 + 64 * slice_align(fm);
  int rc;
  if ((rc = nimfm_comm_alloc(ctx, &fm->pool, (size_t)fm->poolCap)) || (rc = nimfm_comm_alloc(ctx, &fm->grad, (size_t)fm->poolCap))) {
    nimfm_fm_free(ctx, fm);
    return rc;
  }
  fm->P = fm->pool;
  fm->w = fm->pool + nP;
  fm->b = fm->pool + nP + d;
  cudaError_t ce = cudaMalloc(&fm->lams, (size_t)fm->k * 8);
  if (ce == cudaSuccess) ce = cudaMemsetAsync(fm->pool, 0, (size_t)fm->poolCap * 8, ctx->stream);
  if (ce == cudaSuccess) ce = cudaMemsetAsync(fm->grad, 0, (size_t)fm->poolCap * 8, ctx->stream);
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(ctx->stream);
  if (ce != cudaSuccess) {
    nimfm_fm_free(ctx, fm);
    return nimfm_fail(ctx, NIMFM_ERR_CUDA, "nimfm_fm_create: %s", cudaGetErrorString(ce));
  }
  *out = fm;
  return NIMFM_OK;
}

int32_t nimfm_fm_free(nimfm_ctx *ctx, nimfm_fm *fm) {
  if (!fm) return NIMFM_OK;
  if (ctx) cudaSetDevice(ctx->device);
  nimfm_comm_free(ctx, fm->pool);   // P, w, b
  nimfm_comm_free(ctx, fm->grad);
  nimfm_comm_free(ctx, fm->dG);
  nimfm_comm_free(ctx, fm->sgdCnt);
  for (double *p : {fm->lams, fm->gsP, fm->gnP, fm->gsw, fm->gnw,
                    fm->adaScal, fm->scalingsP, fm->scalingsW, fm->sgdScal, fm->Pcm, fm->yPred, fm->Acache,
                    fm->colNormSq, fm->cdScal, fm->proxState, fm->psgdThr})
    cudaFree(p);
  cudaFree(fm->lazyInv);
  cudaFree(fm->lazyFlag);
  delete fm;
  return NIMFM_OK;
}

int32_t nimfm_fm_set_params(nimfm_ctx *ctx, nimfm_fm *fm, const double *P, const double *w, double intercept,
                            const double *lams) {
  if (!ctx || !fm) return NIMFM_ERR_INVALID;
  const int64_t nP = fm->nP();
  REQUIRE((P != nullptr || nP == 0) && w != nullptr, "P / w are NULL");
  CK(cudaSetDevice(ctx->device));
  double *tmp = nullptr;
  if (nP > 0) {
    CK(cudaMalloc(&tmp, (size_t)nP * 8));
    { int rcs = nimfm_staged_h2d(ctx, tmp, P, (size_t)nP * 8); if (rcs) { cudaFree(tmp); return rcs; } }
    permute_model_to_dev<<<ew_grid(ctx, nP), 256, 0, ctx->stream>>>(tmp, fm->P, fm->nOrders, fm->k, fm->dd());
    LAUNCHED(ctx);
  }
  CK(cudaMemcpyAsync(fm->w, w, (size_t)fm->d * 8, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(fm->b, &intercept, 8, cudaMemcpyHostToDevice, ctx->stream));
  fm->lamsAreOnes = true;
  if (lams) {
    for (int s = 0; s < fm->k; s++)
      if (lams[s] != 1.0) fm->lamsAreOnes = false;
    CK(cudaMemcpyAsync(fm->lams, lams, (size_t)fm->k * 8, cudaMemcpyHostToDevice, ctx->stream));
  }
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaFree(tmp));
  CK(cudaGetLastError());
  return NIMFM_OK;
}

static int get_permuted(nimfm_ctx *ctx, nimfm_fm *fm, const double *dev, double *host) {
  const int64_t nP = fm->nP();
  if (nP == 0) return NIMFM_OK;   // degree 1: no P
  double *tmp = nullptr;
  CK(cudaMalloc(&tmp, (size_t)nP * 8));
  permute_dev_to_model<<<ew_grid(ctx, nP), 256, 0, ctx->stream>>>(dev, tmp, fm->nOrders, fm->k, fm->dd());
  LAUNCHED(ctx);
  { int rcs = nimfm_staged_d2h(ctx, host, tmp, (size_t)nP * 8); if (rcs) { cudaFree(tmp); return rcs; } }
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaFree(tmp));
  CK(cudaGetLastError());
  return NIMFM_OK;
}

int32_t nimfm_fm_get_params(nimfm_ctx *ctx, nimfm_fm *fm, double *P, double *w, double *intercept) {
  if (!ctx || !fm) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  if (P) {
    int rc = get_permuted(ctx, fm, fm->P, P);
    if (rc) return rc;
  }
  if (w) CK(cudaMemcpy(w, fm->w, (size_t)fm->d * 8, cudaMemcpyDeviceToHost));
  if (intercept) CK(cudaMemcpy(intercept, fm->b, 8, cudaMemcpyDeviceToHost));
  return NIMFM_OK;
}

int32_t nimfm_fm_get_grads(nimfm_ctx *ctx, nimfm_fm *fm, double *gP, double *gw, double *gb) {
  if (!ctx || !fm) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  const int64_t nP = fm->nP();
  if (gP) {
    int rc = get_permuted(ctx, fm, fm->grad, gP);
    if (rc) return rc;
  }
  if (gw) CK(cudaMemcpy(gw, fm->grad + nP, (size_t)fm->d * 8, cudaMemcpyDeviceToHost));
  if (gb) CK(cudaMemcpy(gb, fm->grad + nP + fm->d, 8, cudaMemcpyDeviceToHost));
  return NIMFM_OK;
}

int32_t nimfm_fm_grad_device_ptr(nimfm_fm *fm, void **ptr, int64_t *nDoubles) {
  if (!fm || !ptr) return NIMFM_ERR_INVALID;
  *ptr = fm->grad;
  if (nDoubles) *nDoubles = fm->nP() + fm->d + 2;
  return NIMFM_OK;
}

// ================================================================== K1: decisionFunction
}  // extern "C"

// device-resident variant used by the CD set-up (cd.nim:144-151): dOut[n] on the device
int nimfm_fm_predict_device(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *Xcsr, double *dOut) {
  int rc = check_fm_ds(ctx, fm, Xcsr, false);
  if (rc) return rc;
  if (Xcsr->n == 0) return NIMFM_OK;
  RowPlan pl;
  if ((rc = plan_rows(ctx, fm, Xcsr, Xcsr->n, MODE_PREDICT, &pl))) return rc;
  RowArgs a;
  fill_row_args(a, fm, Xcsr);
  a.lams = nullptr;   // cd.fit sums A[:, degree-order] without lams (cd.nim:151)
  a.nRows = Xcsr->n;
  a.yOut = dOut;
  a.G = pl.G;
  a.CH = pl.CH;
  pl.kern<<<pl.grid, pl.block, pl.smem, ctx->stream>>>(a);
  LAUNCHED(ctx);
  CK(cudaGetLastError());
  return NIMFM_OK;
}

// decisionFunction's forward (lams applied, factorization_machine.nim:120) into a device buffer
static int nimfm_fm_predict_device_lams(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *Xcsr, double *dOut) {
  int rc = check_fm_ds(ctx, fm, Xcsr, false);
  if (rc) return rc;
  if (Xcsr->n == 0) return NIMFM_OK;
  RowPlan pl;
  if ((rc = plan_rows(ctx, fm, Xcsr, Xcsr->n, MODE_PREDICT, &pl))) return rc;
  RowArgs a;
  fill_row_args(a, fm, Xcsr);
  a.nRows = Xcsr->n;
  a.yOut = dOut;
  a.G = pl.G;
  a.CH = pl.CH;
  pl.kern<<<pl.grid, pl.block, pl.smem, ctx->stream>>>(a);
  LAUNCHED(ctx);
  CK(cudaGetLastError());
  return NIMFM_OK;
}

extern "C" {

int32_t nimfm_fm_decision_function(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, double *out) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(fm && X && out, "NULL argument");
  CK(cudaSetDevice(ctx->device));
  nimfm_dataset *twin = nullptr;
  const nimfm_dataset *Xr = X;
  if (X->kind == NIMFM_DS_CSC) {
    // The ColDataset kernels (kernels.nim:4-11,22-43) visit columns in ascending order, which is the
    // order a CSR row with sorted indices is visited in; run the row kernel on the stable transpose.
    int rc = nimfm_dataset_transpose(ctx, X, &twin);
    if (rc) return rc;
    Xr = twin;
  }
  int rc = check_fm_ds(ctx, fm, Xr, false);
  if (rc) { nimfm_dataset_free(ctx, twin); return rc; }
  const int64_t n = Xr->n;
  if (n == 0) { nimfm_dataset_free(ctx, twin); return NIMFM_OK; }
  RowPlan pl;
  if ((rc = plan_rows(ctx, fm, Xr, n, MODE_PREDICT, &pl))) { nimfm_dataset_free(ctx, twin); return rc; }
  RowKernel kern = pl.kern;
  double *dOut = nullptr;
  CK(cudaMalloc(&dOut, (size_t)n * 8));
  RowArgs a;
  fill_row_args(a, fm, Xr);
  a.rowBegin = 0;
  a.nRows = n;
  a.yOut = dOut;
  a.G = pl.G;
  a.CH = pl.CH;
  kern<<<pl.grid, pl.block, pl.smem, ctx->stream>>>(a);
  LAUNCHED(ctx);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, dOut, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaFree(dOut));
  nimfm_dataset_free(ctx, twin);
  return NIMFM_OK;
}

// ================================================================== K2: predict + grad
// the lazy MBPSGD epoch's view of the pending shrink (RowArgs::lazy*); partialRows returns the number of
// partial rows the kernel wrote (the lazy step reduces them itself: no reduce_partials launch)
struct LazyView {
  double cumPt = 1.0, cumWt = 1.0;
  int64_t partialRows = 0;
};

static int launch_loss_grad(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, int loss, double thr,
                            int64_t rowBegin, int64_t nRows, const int32_t *rowIdxDev, double mb,
                            double *yOutDev, LazyView *lazy = nullptr) {
  RowPlan pl;
  int rc;
  // NIMFM_DETERMINISTIC=1: the atomic-free route (fm_cols.cu): stash-forward row kernel + column kernel over the CSC twin
  if (const char *env = getenv("NIMFM_DETERMINISTIC"); env && env[0] == '1' && !lazy) {
    if (rowIdxDev) return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "the deterministic gradient needs a contiguous row range (no row list)");
    if ((rc = plan_rows(ctx, fm, X, nRows, MODE_STASH, &pl))) return rc;
    RowArgs base;
    fill_row_args(base, fm, X);
    return nimfm_fm_det_loss_grad(ctx, fm, X, pl, loss, thr, rowBegin, nRows, mb, yOutDev, base);
  }
  rc = plan_rows(ctx, fm, X, nRows, MODE_GRAD, &pl);
  if (rc) return rc;
  if (lazy && !pl.stream) return nimfm_fail(ctx, NIMFM_ERR_STATE, "lazy step without the streaming row kernel");
  RowKernel kern = pl.kern;
  if ((rc = nimfm_ensure_partials(ctx, (size_t)pl.nWarps * 4))) return rc;
  RowArgs a;
  fill_row_args(a, fm, X);
  a.rowBegin = rowBegin;
  a.nRows = nRows;
  a.rowIdx = rowIdxDev;
  a.yOut = yOutDev;
  a.gP = fm->grad;
  a.gw = fm->grad + fm->nP();
  a.partials = ctx->partials;
  a.loss = loss;
  a.thr = thr;
  a.mb = mb;
  a.G = pl.G;
  a.CH = pl.CH;
  if (lazy) {
    a.lazyInv = fm->lazyInv;
    a.lazyFlag = fm->lazyFlag;
    a.lazyCumPt = lazy->cumPt;
    a.lazyCumWt = lazy->cumWt;
    lazy->partialRows = pl.nWarps;
  }
  kern<<<pl.grid, pl.block, pl.smem, ctx->stream>>>(a);
  LAUNCHED(ctx);
  if (lazy) return NIMFM_OK;
  // tail += [sum coef, sum loss]: partial columns are (loss, coef, dL^2, viol) -> reorder via scratch
  reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(ctx->partials, pl.nWarps, ctx->scalars + 8, 0);
  LAUNCHED(ctx);
  return NIMFM_OK;
}

// The gradient of one minibatch of the MBPSGD and minibatch-SGD epochs (rows rowIdxDev[0 .. nRows), or the cursor
// (rowBegin + q) mod n) into fm->grad, red4 at ctx->scalars + 8.  Under NIMFM_DETERMINISTIC=1 a row list or a cursor
// that wraps past the last row cannot clip the dataset's column twin to a row range, so such a minibatch gets its own
// column index (nimfm_mb_index_build) and the stash forward and column kernel run over its view; red4 is summed from
// the rows' decision values (FmDetTargets::yhat), so the tuned and the generic forms give the same bits.  Every other
// minibatch takes launch_loss_grad as before.
static int minibatch_loss_grad(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, int loss, double thr,
                               int64_t rowBegin, int64_t nRows, const int32_t *rowIdxDev, double mb) {
  const char *env = getenv("NIMFM_DETERMINISTIC");
  if (!(env && env[0] == '1') || (!rowIdxDev && rowBegin + nRows <= X->n))
    return launch_loss_grad(ctx, fm, X, loss, thr, rowBegin, nRows, rowIdxDev, mb, nullptr);
  nimfm_trace_begin(ctx, "det index");
  nimfm_mb_index *ix = nullptr;
  int rc = nimfm_mb_index_build(ctx, X, fm->nAug, rowBegin, nRows, rowIdxDev, &ix);
  nimfm_trace_end(ctx);
  if (rc) return rc;
  nimfm_trace_begin(ctx, "det passes");
  RowPlan pl;
  rc = plan_rows(ctx, fm, &ix->view, nRows, MODE_STASH, &pl);
  if (!rc) {
    RowArgs base;
    fill_row_args(base, fm, &ix->view);
    FmDetTargets o;
    o.gP = fm->grad;
    o.gw = fm->grad + fm->nP();
    o.red4 = ctx->scalars + 8;
    o.yhat = ix->yhat;
    rc = nimfm_fm_det_pass(ctx, fm, &ix->tw, pl, loss, thr, 0, nRows, mb, nullptr, base, o);
  }
  nimfm_trace_end(ctx);
  return rc;
}


int32_t nimfm_fm_loss_grad(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, int32_t loss,
                           double huberThreshold, int64_t rowBegin, int64_t nRows, const int64_t *rowIdx,
                           int64_t miniBatchSize, int32_t zeroGrads, int32_t allreduce, double *lossSum) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int rc = check_fm_ds(ctx, fm, X, true);
  if (rc) return rc;
  REQUIRE(nRows >= 0 && miniBatchSize >= 1, "bad nRows / miniBatchSize");
  REQUIRE(rowIdx != nullptr || (rowBegin >= 0 && (rowBegin < X->n || nRows == 0)), "rowBegin out of range");
  const int64_t nG = fm->nP() + fm->d + 2;
  PeerScope peers(ctx, {allreduce ? fm->grad : nullptr});   // collective when a communicator exists: all ranks call together
  if (peers.rc) return peers.rc;
  if (zeroGrads) CK(cudaMemsetAsync(fm->grad, 0, (size_t)nG * 8, ctx->stream));
  const int32_t *idxDev = nullptr;
  if (rowIdx && nRows > 0) {
    if ((rc = nimfm_stage_row_ids(ctx, rowIdx, nRows, X->n))) return rc;
    idxDev = ctx->idx32Scratch;
  }
  if (nRows > 0) {
    if ((rc = launch_loss_grad(ctx, fm, X, loss, huberThreshold, rowBegin, nRows, idxDev, (double)miniBatchSize, nullptr)))
      return rc;
    add_tail_kernel<<<1, 1, 0, ctx->stream>>>(fm->grad + nG - 2, ctx->scalars + 8);
    LAUNCHED(ctx);
  }
  if (allreduce && (rc = nimfm_allreduce_sum(ctx, fm->grad, nG))) return rc;
  CK(cudaGetLastError());
  if (lossSum) CK(cudaMemcpyAsync(lossSum, fm->grad + nG - 1, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return NIMFM_OK;
}

int32_t nimfm_fm_time_loss_grad(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, int32_t loss,
                                int64_t nRows, int64_t miniBatchSize, int32_t reps, int32_t gradToo,
                                float *msPerLaunch) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int rc = check_fm_ds(ctx, fm, X, gradToo != 0);
  if (rc) return rc;
  REQUIRE(reps >= 1 && nRows >= 1 && msPerLaunch, "bad arguments");
  RowPlan pl;
  if ((rc = plan_rows(ctx, fm, X, nRows, gradToo ? MODE_GRAD : MODE_PREDICT, &pl))) return rc;
  RowKernel kern = pl.kern;
  if ((rc = nimfm_ensure_partials(ctx, (size_t)pl.nWarps * 4))) return rc;
  double *dOut = nullptr;
  if (!gradToo) CK(cudaMalloc(&dOut, (size_t)nRows * 8));
  RowArgs a;
  fill_row_args(a, fm, X);
  a.nRows = nRows;
  a.yOut = dOut;
  a.gP = fm->grad;
  a.gw = fm->grad + fm->nP();
  a.partials = ctx->partials;
  a.loss = loss;
  a.thr = 1.0;
  a.mb = (double)miniBatchSize;
  a.G = pl.G;
  a.CH = pl.CH;
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  for (int r = 0; r < reps; r++) {
    kern<<<pl.grid, pl.block, pl.smem, ctx->stream>>>(a);
    LAUNCHED(ctx);
  }
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  CK(cudaEventSynchronize(ctx->ev1));
  CK(cudaGetLastError());
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
  *msPerLaunch = ms / reps;
  if (dOut) CK(cudaFree(dOut));
  return NIMFM_OK;
}

// ================================================================== MBPSGD epoch (minibatch_psgd.nim:91-124)
static double get_eta(int sched, double eta0, double power, double reg, int64_t it) {  // sgd.nim:60-69
  switch (sched) {
    case NIMFM_SCHED_CONSTANT: return eta0;
    case NIMFM_SCHED_OPTIMAL: return eta0 / pow(1.0 + eta0 * reg * (double)it, power);
    case NIMFM_SCHED_INVSCALING: return eta0 / pow((double)it, power);
    default: return 1.0 / (reg * (double)it);
  }
}

// reg.prox(params.P[order], lam, degree-order) for every order (minibatch_psgd.nim:119-121), for the
// regularisers the dense step kernel does not fuse (L1 is fused there).  Enqueued on ctx->stream; the
// column-wise SquaredL12 iterates to its fixed point with a host check every few sweeps.
static int apply_prox(nimfm_ctx *ctx, nimfm_fm *fm, int reg, double lam) {
  if (reg == NIMFM_REG_IDENTITY || reg == NIMFM_REG_L1 || lam == 0.0 || fm->nOrders == 0) return NIMFM_OK;   // degree 1: no P to prox
  const int64_t dd = fm->dd();
  const int SB8 = fm->nOrders * fm->k;
  if (reg == NIMFM_REG_L21 || reg == NIMFM_REG_SQUAREDL12_ROWS) {
    if (fm->k > 32 * NIMFM_PROX_MAXE)
      return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "row-wise prox supports nComponents <= %d", 32 * NIMFM_PROX_MAXE);
    const int64_t nRows = dd * fm->nOrders;
    prox_rows_kernel<<<ew_grid(ctx, nRows * 32), 256, 0, ctx->stream>>>(fm->P, nRows, fm->k, lam, reg);
    LAUNCHED(ctx);
    return NIMFM_OK;
  }
  if (reg != NIMFM_REG_SQUAREDL12) return nimfm_fail(ctx, NIMFM_ERR_INVALID, "unknown regulariser %d", reg);
  if (SB8 > 1024) return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "nOrders*nComponents=%d > 1024", SB8);
  const int R = std::max(1, 256 / SB8), block = R * SB8;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((dd + R - 1) / R, (int64_t)ctx->numSMs * 8));
  int rc = nimfm_ensure_partials(ctx, (size_t)grid * SB8 * 2);
  if (rc) return rc;
  if (!fm->proxState) CK(cudaMalloc(&fm->proxState, (size_t)(3 * SB8 + 8) * 8));
  sql12_init_kernel<<<1, 256, 0, ctx->stream>>>(fm->proxState, SB8);
  LAUNCHED(ctx);
  bool done = false;
  for (int iter = 0; iter < 1024 && !done; ++iter) {
    sql12_pass_kernel<<<grid, block, (size_t)block * 16, ctx->stream>>>(fm->P, dd, SB8, R, fm->proxState, ctx->partials);
    sql12_update_kernel<<<1, 256, 0, ctx->stream>>>(ctx->partials, grid, SB8, lam, fm->proxState);
    ctx->launches += 2;
    if ((iter & 3) == 3) {
      CK(cudaMemcpyAsync(ctx->hostScalars + 8, fm->proxState + 3 * SB8, 8, cudaMemcpyDeviceToHost, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));
      done = ctx->hostScalars[8] != 0.0;
    }
  }
  if (!done) return nimfm_fail(ctx, NIMFM_ERR_STATE, "SquaredL12 prox did not reach its fixed point");
  sql12_apply_kernel<<<grid, block, 0, ctx->stream>>>(fm->P, dd, SB8, R, fm->proxState);
  LAUNCHED(ctx);
  return NIMFM_OK;
}

// entry points for psgd.cu (the SquaredL12 route of PSGD reuses the row kernel and the prox kernels)
int nimfm_fm_apply_prox(nimfm_ctx *ctx, nimfm_fm *fm, int reg, double lam) { return apply_prox(ctx, fm, reg, lam); }
// the gradient of rows of a resident dataset into fm->grad (+ red4 at ctx->scalars+8), for sgd_mb.cu
int nimfm_fm_launch_grad_rows(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, int loss, double thr,
                              int64_t rowBegin, int64_t nRows, const int32_t *rowIdxDev, double mb) {
  return minibatch_loss_grad(ctx, fm, X, loss, thr, rowBegin, nRows, rowIdxDev, mb);
}
double nimfm_get_eta(int sched, double eta0, double power, double reg, int64_t it) { return get_eta(sched, eta0, power, reg, it); }
int nimfm_fm_loss_grad_one_row(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, int loss, double thr,
                               int64_t row) {
  int rc = launch_loss_grad(ctx, fm, X, loss, thr, row, 1, nullptr, 1.0, nullptr);
  if (rc) return rc;
  add_tail_kernel<<<1, 1, 0, ctx->stream>>>(fm->grad + fm->nP() + fm->d, ctx->scalars + 8);
  LAUNCHED(ctx);
  return NIMFM_OK;
}

int32_t nimfm_fm_mbpsgd_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_mbpsgd_cfg *cfg,
                              int64_t localBatch, int64_t *it, int64_t *ii, const int64_t *sampleIdx,
                              double *runningLoss) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int rc = check_fm_ds(ctx, fm, X, true);
  if (rc) return rc;
  REQUIRE(cfg && it && ii, "NULL argument");
  REQUIRE(cfg->miniBatchSize >= 1 && cfg->maxIterInner >= 1, "miniBatchSize / maxIterInner must be resolved (>= 1)");
  REQUIRE(cfg->reg >= NIMFM_REG_IDENTITY && cfg->reg <= NIMFM_REG_L21, "unsupported regulariser");
  // SquaredL12.initSGD raises for degree != 2 (squaredl12.nim:103-106)
  REQUIRE(!((cfg->reg == NIMFM_REG_SQUAREDL12 || cfg->reg == NIMFM_REG_SQUAREDL12_ROWS) && fm->degree != 2),
          "SquaredL12 supports only degree=2.");
  if (localBatch <= 0) localBatch = cfg->miniBatchSize;
  REQUIRE(X->n > 0, "empty dataset");
  if (ctx->nranks > 1) {
    // every rank must run the same number of minibatches with the same divisor and step sizes, and the shares
    // must add up to the global minibatch -- otherwise the collectives deadlock or the replicas drift apart
    const int64_t mine[4] = {cfg->miniBatchSize, cfg->maxIterInner, localBatch, *it};
    std::vector<int64_t> all((size_t)4 * ctx->nranks);
    if ((rc = nimfm_allgather_host_i64(ctx, mine, 4, all.data()))) return rc;
    int64_t share = 0;
    for (int r = 0; r < ctx->nranks; r++) {
      const int64_t *q = all.data() + 4 * r;
      REQUIRE(q[0] == mine[0] && q[1] == mine[1] && q[3] == mine[3],
              "rank %d disagrees on miniBatchSize / maxIterInner / it (%lld, %lld, %lld vs %lld, %lld, %lld)", r,
              (long long)q[0], (long long)q[1], (long long)q[3], (long long)mine[0], (long long)mine[1], (long long)mine[3]);
      share += q[2];
    }
    REQUIRE(share == cfg->miniBatchSize, "the ranks' localBatch add up to %lld, not miniBatchSize %lld", (long long)share,
            (long long)cfg->miniBatchSize);
  }
  const int64_t nP = fm->nP(), d = fm->d, nG = nP + d + 2;
  PeerScope peers(ctx, {fm->grad, fm->pool});
  if (peers.rc) return peers.rc;
  const int64_t total = localBatch * cfg->maxIterInner;
  const int32_t *idxDev = nullptr;
  if (sampleIdx) {
    if ((rc = nimfm_stage_row_ids(ctx, sampleIdx, total, X->n))) return rc;
    idxDev = ctx->idx32Scratch;
  }
  CK(cudaMemsetAsync(fm->grad, 0, (size_t)nG * 8, ctx->stream));       // grads <- 0 (:99)
  CK(cudaMemsetAsync(ctx->scalars, 0, 8, ctx->stream));
  int64_t cur = *ii;
  // ---- lazy epoch (dense_kernels.cuh, K3b): one rank, no prox, minibatches that touch a minority of the
  // features.  Same iterates as the dense step up to the rounding of the accumulated shrink factors.
  {
    const int64_t T = cfg->maxIterInner;
    const bool noProx = cfg->reg == NIMFM_REG_IDENTITY || cfg->gamma == 0.0;   // lam = 0: every prox is the identity
    const char *env = getenv("NIMFM_MBPSGD_LAZY");
    const double touchedUpper = (double)localBatch * ((double)X->nnz / (double)X->n + fm->nAug);
    bool lazy = ctx->nranks == 1 && noProx && T >= 2 && T < (1 << 30) && touchedUpper <= 2.0 * (double)fm->dd();   // measured crossover on the C3 shape: between 1.3 and 5 nnz per feature
    if (env) lazy = env[0] == '1' && ctx->nranks == 1 && noProx && T < (1 << 30);
    if (const char *det = getenv("NIMFM_DETERMINISTIC"); det && det[0] == '1') lazy = false;   // the lazy step folds factors into x: RED route only
    RowPlan plq;
    if (lazy && (plan_rows(ctx, fm, X, localBatch, MODE_GRAD, &plq) != NIMFM_OK || !plq.stream)) lazy = false;
    { const int sb = fm->nOrders * fm->k; if (sb & (sb - 1)) lazy = false; }   // the flat step shifts by log2(SB8)
    std::vector<double> cum;
    if (lazy) {   // cumulative shrink tables cum[t] = prod_{s<t} 1 / (1 + eta_s * reg); too small a product: dense
      cum.assign(2 * (size_t)(T + 1), 1.0);
      for (int64_t t = 0; t < T; t++) {
        const double etaP = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->beta, *it + t);
        const double etaW = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha, *it + t);
        cum[t + 1] = cum[t] * (1.0 / (1.0 + etaP * cfg->beta));
        // fitLinear = false: w is frozen (params.nim:90-98), and the row kernel must see it unscaled
        cum[T + 1 + t + 1] = fm->fitLinear ? cum[T + 1 + t] * (1.0 / (1.0 + etaW * cfg->alpha)) : 1.0;
      }
      if (!(cum[T] > 1e-100) || !(cum[2 * T + 1] > 1e-100)) lazy = false;
    }
    if (lazy) {
      const int64_t dd = fm->dd();
      const int SB8 = fm->nOrders * fm->k;
      int shift = 0;
      while ((1 << shift) < SB8) shift++;
      if (!fm->lazyInv) {
        CK(cudaMalloc(&fm->lazyInv, (size_t)dd * sizeof(double2)));
        CK(cudaMalloc(&fm->lazyFlag, (size_t)dd));
        CK(cudaMemsetAsync(fm->lazyFlag, 0, (size_t)dd, ctx->stream));
        mbpsgd_lazy_flush_feat_kernel<<<ew_grid(ctx, dd), 256, 0, ctx->stream>>>(nullptr, 0, 0, fm->lazyInv, dd, 1.0);
        LAUNCHED(ctx);
      }
      const int grid = ctx->numSMs * 8;
      for (int64_t inner = 0; inner < T; inner++) {
        LazyView lv;
        lv.cumPt = cum[inner];
        lv.cumWt = cum[T + 1 + inner];
        if ((rc = launch_loss_grad(ctx, fm, X, cfg->loss, cfg->huberThreshold, cur, localBatch,
                                   idxDev ? idxDev + inner * localBatch : nullptr, (double)cfg->miniBatchSize, nullptr, &lv)))
          return rc;
        const double etaP = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->beta, *it);
        const double etaW = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha, *it);
        const double etaB = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha0, *it);
        const double rP = 1.0 / (1.0 + etaP * cfg->beta), rW = 1.0 / (1.0 + etaW * cfg->alpha),
                     rB = 1.0 / (1.0 + etaB * cfg->alpha0);
        mbpsgd_lazy_step_kernel<<<grid, 256, 0, ctx->stream>>>(
            fm->P, fm->grad, shift, dd, d, fm->w, fm->grad + nP, fm->lazyFlag, fm->lazyInv, lv.cumPt, lv.cumWt,
            1.0 / cum[inner + 1], 1.0 / cum[T + 1 + inner + 1], -etaP, rP, 1.0, -etaW, rW, 1.0, fm->fitLinear, fm->b,
            ctx->partials, lv.partialRows, -etaB, rB, fm->fitIntercept, ctx->scalars, nullptr);
        LAUNCHED(ctx);
        *it += 1;
        cur = (cur + localBatch) % X->n;
      }
      mbpsgd_lazy_flush_P_kernel<<<ew_grid(ctx, nP), 256, 0, ctx->stream>>>(fm->P, shift, nP, fm->lazyInv, cum[T]);
      LAUNCHED(ctx);
      mbpsgd_lazy_flush_feat_kernel<<<ew_grid(ctx, dd), 256, 0, ctx->stream>>>(fm->w, d, fm->fitLinear, fm->lazyInv, dd,
                                                                             cum[2 * T + 1]);
      LAUNCHED(ctx);
      CK(cudaGetLastError());
      CK(cudaMemcpyAsync(ctx->hostScalars, ctx->scalars, 8, cudaMemcpyDeviceToHost, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));
      *ii = cur;
      if (runningLoss) *runningLoss = ctx->hostScalars[0] / (double)(cfg->miniBatchSize * cfg->maxIterInner);
      return NIMFM_OK;
    }
  }
  // ---- multi-rank, sharded step (SURVEY 8e, the alternative to "identical dense step on every GPU"): every rank
  // owns a flat 1/N slice of [P | w | b]; the gradient pool is reduced slice-wise, the owner steps (and proxes) its
  // slice, and the slice is distributed to all ranks.  Over NVLink peer memory (peer.cu) that is ONE kernel between
  // two flag barriers -- reduce out of every peer's gradient pool, Params.step + L1 prox, stores into every peer's
  // parameter pool -- in a fixed rank order; without peer mapping (NIMFM_PEER=0, no P2P) NCCL carries it as an
  // all-reduce + the dense step everywhere, or (NIMFM_MBPSGD_SHARDED=1) reduce-scatter -> slice step -> all-gather.
  // The column-wise SquaredL12 prox needs sums over all features and keeps the all-reduce + dense step.
  int64_t sliceC = 0;
  bool viaPeer = false;
  {
    const char *envS = getenv("NIMFM_MBPSGD_SHARDED");
    const int64_t align = slice_align(fm);
    const int64_t c = ((nG + ctx->nranks - 1) / ctx->nranks + align - 1) / align * align;
    const bool fits = ctx->nranks > 1 && cfg->reg != NIMFM_REG_SQUAREDL12 && c * ctx->nranks <= fm->poolCap;
    viaPeer = fits && ctx->peerOK && !(envS && envS[0] == '0');
    if (viaPeer || (fits && envS && envS[0] == '1')) sliceC = c;
  }
  if (sliceC) CK(cudaMemsetAsync(fm->b + 1, 0, 8, ctx->stream));   // epoch loss slot of the parameter pool
  for (int64_t inner = 0; inner < cfg->maxIterInner; inner++) {
    nimfm_trace_begin(ctx, "K2");
    if ((rc = minibatch_loss_grad(ctx, fm, X, cfg->loss, cfg->huberThreshold, cur, localBatch,
                                  idxDev ? idxDev + inner * localBatch : nullptr, (double)cfg->miniBatchSize)))
      return rc;
    add_tail_kernel<<<1, 1, 0, ctx->stream>>>(fm->grad + nG - 2, ctx->scalars + 8);
    LAUNCHED(ctx);
    nimfm_trace_end(ctx);
    if (sliceC) {
      const double etaP = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->beta, *it);
      const double etaW = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha, *it);
      const double etaB = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha0, *it);
      const double rP = 1.0 / (1.0 + etaP * cfg->beta), rW = 1.0 / (1.0 + etaW * cfg->alpha),
                   rB = 1.0 / (1.0 + etaB * cfg->alpha0);
      const double lam = cfg->gamma * etaP / (1.0 + etaP * cfg->beta);
      const int64_t lo = std::min(nG, (int64_t)ctx->rank * sliceC), hi = std::min(lo + sliceC, nG);
      const bool rowProx = (cfg->reg == NIMFM_REG_L21 || cfg->reg == NIMFM_REG_SQUAREDL12_ROWS) && lam != 0.0;
      if (rowProx && fm->k > 32 * NIMFM_PROX_MAXE)
        return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "row-wise prox supports nComponents <= %d", 32 * NIMFM_PROX_MAXE);
      auto prox_slice = [&]() {   // whole (feature, order) vectors: slices start at multiples of nOrders*k
        if (!rowProx || lo >= nP) return;
        const int64_t vecs = (std::min(hi, nP) - lo) / fm->k;
        prox_rows_kernel<<<ew_grid(ctx, vecs * 32), 256, 0, ctx->stream>>>(fm->pool + lo, vecs, fm->k, lam, cfg->reg);
        LAUNCHED(ctx);
      };
      int done = 0;
      if (viaPeer) {
        MbpsgdStepArgs sa{nP, d, -etaP, rP, lam, -etaW, rW, -etaB, rB, cfg->reg, fm->fitLinear, fm->fitIntercept};
        nimfm_trace_begin(ctx, "barrier+reduce+step");
        if ((rc = nimfm_peer_mbpsgd_step(ctx, fm->pool, fm->grad, lo, hi, sa, &done))) return rc;
        nimfm_trace_end(ctx);
        if (done) {
          prox_slice();
          nimfm_trace_begin(ctx, "barrier2");
          if ((rc = nimfm_peer_barrier(ctx))) return rc;   // every slice is final; all peers are done reading my gradients
          nimfm_trace_end(ctx);
          // the pull first, grads <- 0 last.  Measured on 2 GPUs (C3, 256 Ki rows per rank per minibatch,
          // profiles/r02_peer_exchange.md): with the pull last, the rank whose pulled slice holds the always-present
          // columns' parameter rows ran the next row kernel at 740 us against 598 us on the other rank (freshly
          // written hot lines, whoever wrote them); with the zero-fill last both ranks run it at 630-646 us
          nimfm_trace_begin(ctx, "pull");
          if ((rc = nimfm_peer_pull_slices(ctx, fm->pool, sliceC, nG))) return rc;
          nimfm_trace_end(ctx);
          nimfm_trace_begin(ctx, "zero grads");
          fill_kernel<<<ew_grid(ctx, nG), 256, 0, ctx->stream>>>(fm->grad, nG, 0.0);
          LAUNCHED(ctx);
          nimfm_trace_end(ctx);
          *it += 1;
          cur = (cur + localBatch) % X->n;
          continue;
        }
      }
      if (!done) {
        if ((rc = nimfm_reduce_scatter_sum(ctx, fm->grad, sliceC))) return rc;
        if (hi > lo) {
          mbpsgd_step_flat_kernel<<<ew_grid(ctx, hi - lo), 256, 0, ctx->stream>>>(
              fm->pool, fm->grad, lo, hi, nP, d, -etaP, rP, cfg->reg, lam, -etaW, rW, fm->fitLinear, -etaB, rB,
              fm->fitIntercept);
          LAUNCHED(ctx);
          prox_slice();
        }
        if ((rc = nimfm_allgather_inplace(ctx, fm->pool, sliceC))) return rc;
      }
      // grads <- 0 by a kernel, not a memset: its stores leave the lines in L2 for the next minibatch's REDs
      nimfm_trace_begin(ctx, "zero grads");
      fill_kernel<<<ew_grid(ctx, sliceC * ctx->nranks), 256, 0, ctx->stream>>>(fm->grad, sliceC * ctx->nranks, 0.0);
      LAUNCHED(ctx);
      nimfm_trace_end(ctx);
      *it += 1;
      cur = (cur + localBatch) % X->n;
      continue;
    }
    nimfm_trace_begin(ctx, "allreduce");
    if ((rc = nimfm_allreduce_sum(ctx, fm->grad, nG))) return rc;
    nimfm_trace_end(ctx);
    nimfm_trace_begin(ctx, "dense step");
    struct TraceEnd { nimfm_ctx *c; ~TraceEnd() { nimfm_trace_end(c); } } traceEnd{ctx};
    const double etaP = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->beta, *it);     // :114-116
    const double etaW = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha, *it);
    const double etaB = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha0, *it);
    const double rP = 1.0 / (1.0 + etaP * cfg->beta), rW = 1.0 / (1.0 + etaW * cfg->alpha),
                 rB = 1.0 / (1.0 + etaB * cfg->alpha0);
    const double lam = cfg->gamma * etaP / (1.0 + etaP * cfg->beta);                         // :119-121
    mbpsgd_step_kernel<<<ew_grid(ctx, std::max(nP, d)), 256, 0, ctx->stream>>>(
        fm->P, fm->grad, nP, -etaP, rP, cfg->reg, lam, fm->w, fm->grad + nP, d, -etaW, rW, fm->fitLinear, fm->b,
        fm->grad + nG - 2, -etaB, rB, fm->fitIntercept, ctx->scalars);
    LAUNCHED(ctx);
    if ((rc = apply_prox(ctx, fm, cfg->reg, lam))) return rc;
    *it += 1;
    cur = (cur + localBatch) % X->n;
  }
  if (viaPeer && (rc = nimfm_peer_barrier(ctx))) return rc;   // no peer still pulls my slice when the call returns
  CK(cudaGetLastError());
  nimfm_trace_report(ctx, "mbpsgd epoch");
  CK(cudaMemcpyAsync(ctx->hostScalars, sliceC ? fm->b + 1 : ctx->scalars, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *ii = cur;
  // runningLoss / (miniBatchSize*maxIterInner) (:124); the loss sum was reduced with the gradient
  if (runningLoss) *runningLoss = ctx->hostScalars[0] / (double)(cfg->miniBatchSize * cfg->maxIterInner);
  return NIMFM_OK;
}

// ================================================================== minibatch SGD, lazy form (sgd_mb.cu, K6b)
// The rule of sgd_mb.cu with the K3b machinery: untouched features owe cum[t] * inv[j] = prod (1-eta beta)^B of
// the minibatches they sat out; the row kernel folds it into x, two flat kernels update the touched features,
// one dense pass at the end of the epoch settles the rest.  *applied = 0: not applicable here (the caller runs
// the dense form).  idxDev: staged sample order (nullable).
int nimfm_fm_sgd_mb_lazy_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_sgd_cfg *cfg,
                               int64_t B, int64_t *it, const int32_t *idxDev, int64_t nRows, int *applied,
                               double *viol, double *lossSum) {
  *applied = 0;
  if (nRows <= 0 || X->n <= 0) return NIMFM_OK;
  const int64_t T = (nRows + B - 1) / B;
  const char *env = getenv("NIMFM_SGD_MB_LAZY");
  const double touchedUpper = (double)B * ((double)X->nnz / (double)X->n + fm->nAug);
  // measured on the C4 shape: 4 096-row minibatches 11.6 -> 26.4 M samples/s, 65 536-row 73.7 (dense) vs 61.7 (lazy)
  bool lazy = ctx->nranks == 1 && T >= 2 && T < (1 << 30) && touchedUpper <= 2.0 * (double)fm->dd();
  if (env) lazy = env[0] == '1' && ctx->nranks == 1 && T < (1 << 30);
  if (const char *det = getenv("NIMFM_DETERMINISTIC"); det && det[0] == '1') lazy = false;   // the lazy step folds factors into x: RED route only
  const int SB8 = fm->nOrders * fm->k;
  if (SB8 < 1 || (SB8 & (SB8 - 1))) lazy = false;
  RowPlan plq;
  if (lazy && (plan_rows(ctx, fm, X, std::min(B, nRows), MODE_GRAD, &plq) != NIMFM_OK || !plq.stream)) lazy = false;
  if (!lazy) return NIMFM_OK;
  // per-minibatch step sizes / shrink factors and their running products
  std::vector<double> etaP((size_t)T), etaW((size_t)T), etaB((size_t)T), sP((size_t)T), sW((size_t)T), sB((size_t)T);
  std::vector<double> cumP((size_t)T + 1, 1.0), cumW((size_t)T + 1, 1.0);
  auto shrink_pow = [](double base, int64_t n) { double s = 1.0; for (int64_t i = 0; i < n; i++) s *= base; return s; };
  for (int64_t t = 0; t < T; t++) {
    const int64_t Bm = std::min(B, nRows - t * B), itT = *it + t * B;
    etaP[t] = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->beta, itT);
    etaW[t] = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha, itT);
    etaB[t] = get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha0, itT);
    sP[t] = shrink_pow(1.0 - etaP[t] * cfg->beta, Bm);
    sW[t] = shrink_pow(1.0 - etaW[t] * cfg->alpha, Bm);
    sB[t] = shrink_pow(1.0 - etaB[t] * cfg->alpha0, Bm);
    cumP[t + 1] = cumP[t] * sP[t];
    cumW[t + 1] = fm->fitLinear ? cumW[t] * sW[t] : 1.0;   // fitLinear = false: w is frozen and read unscaled
  }
  // a factor that is not a healthy positive number (eta * reg >= 1, long decay): dense form
  if (!(cumP[T] > 1e-100) || !(cumW[T] > 1e-100) || !(cumP[T] < 1e100) || !(cumW[T] < 1e100)) return NIMFM_OK;
  for (int64_t t = 0; t < T; t++)
    if (!(sP[t] > 0.0) || !(sW[t] > 0.0)) return NIMFM_OK;
  const int64_t nP = fm->nP(), d = fm->d, dd = fm->dd(), nG = nP + d + 2;
  int shift = 0;
  while ((1 << shift) < SB8) shift++;
  if (!fm->lazyInv) {
    CK(cudaMalloc(&fm->lazyInv, (size_t)dd * sizeof(double2)));
    CK(cudaMalloc(&fm->lazyFlag, (size_t)dd));
    CK(cudaMemsetAsync(fm->lazyFlag, 0, (size_t)dd, ctx->stream));
    mbpsgd_lazy_flush_feat_kernel<<<ew_grid(ctx, dd), 256, 0, ctx->stream>>>(nullptr, 0, 0, fm->lazyInv, dd, 1.0);
    LAUNCHED(ctx);
  }
  const int grid = ctx->numSMs * 8;
  int rc;
  if ((rc = nimfm_ensure_partials(ctx, (size_t)(plq.nWarps + grid) * 4))) return rc;
  CK(cudaMemsetAsync(fm->grad, 0, (size_t)nG * 8, ctx->stream));
  CK(cudaMemsetAsync(ctx->scalars, 0, 8, ctx->stream));
  CK(cudaMemsetAsync(ctx->scalars + 20, 0, 4 * 8, ctx->stream));
  *applied = 1;
  for (int64_t t = 0; t < T; t++) {
    const int64_t q0 = t * B, Bm = std::min(B, nRows - q0);
    LazyView lv;
    lv.cumPt = cumP[t];
    lv.cumWt = cumW[t];
    if ((rc = launch_loss_grad(ctx, fm, X, cfg->loss, cfg->huberThreshold, q0, Bm, idxDev ? idxDev + q0 : nullptr, 1.0,
                               nullptr, &lv)))
      return rc;
    double *violPart = ctx->partials + (size_t)lv.partialRows * 4;
    mbpsgd_lazy_step_kernel<<<grid, 256, 0, ctx->stream>>>(
        fm->P, fm->grad, shift, dd, d, fm->w, fm->grad + nP, fm->lazyFlag, fm->lazyInv, lv.cumPt, lv.cumWt,
        1.0 / cumP[t + 1], 1.0 / cumW[t + 1], -etaP[t], 1.0, sP[t], -etaW[t], 1.0, sW[t], fm->fitLinear, fm->b,
        ctx->partials, lv.partialRows, -etaB[t], sB[t], fm->fitIntercept, ctx->scalars, violPart);
    LAUNCHED(ctx);
    reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(violPart, grid, ctx->scalars + 20, 1);
    LAUNCHED(ctx);
    *it += Bm;
  }
  mbpsgd_lazy_flush_P_kernel<<<ew_grid(ctx, nP), 256, 0, ctx->stream>>>(fm->P, shift, nP, fm->lazyInv, cumP[T]);
  LAUNCHED(ctx);
  mbpsgd_lazy_flush_feat_kernel<<<ew_grid(ctx, dd), 256, 0, ctx->stream>>>(fm->w, d, fm->fitLinear, fm->lazyInv, dd, cumW[T]);
  LAUNCHED(ctx);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ctx->hostScalars, ctx->scalars, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(ctx->hostScalars + 1, ctx->scalars + 20, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (lossSum) *lossSum = ctx->hostScalars[0];
  if (viol) *viol = ctx->hostScalars[1];
  return NIMFM_OK;
}

// ================================================================== AdaGrad (adagrad.nim)
int32_t nimfm_fm_adagrad_init(nimfm_ctx *ctx, nimfm_fm *fm, double eps, int32_t reset) {
  if (!ctx || !fm) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  const int64_t nP = fm->nP(), d = fm->d, dd = fm->dd();
  const bool fresh = !fm->gsw;   // (not gsP: degree 1 has no P state)
  if (fresh) {
    if (nP > 0) {
      CK(cudaMalloc(&fm->gsP, (size_t)nP * 8));
      CK(cudaMalloc(&fm->gnP, (size_t)nP * 8));
    }
    CK(cudaMalloc(&fm->gsw, (size_t)d * 8));
    CK(cudaMalloc(&fm->gnw, (size_t)d * 8));
    { int rca = nimfm_comm_alloc(ctx, &fm->dG, (size_t)(2 * nP + 2 * d + dd + 8)); if (rca) return rca; }
    CK(cudaMalloc(&fm->adaScal, 8 * 8));
  }
  if (fresh || reset) {   // AdaGrad.init, :47-55
    if (nP > 0) {
      CK(cudaMemsetAsync(fm->gsP, 0, (size_t)nP * 8, ctx->stream));
      fill_kernel<<<ew_grid(ctx, nP), 256, 0, ctx->stream>>>(fm->gnP, nP, eps);
      LAUNCHED(ctx);
    }
    CK(cudaMemsetAsync(fm->gsw, 0, (size_t)d * 8, ctx->stream));
    fill_kernel<<<ew_grid(ctx, d), 256, 0, ctx->stream>>>(fm->gnw, d, eps);
    LAUNCHED(ctx);
    const double sc[2] = {0.0, eps};
    CK(cudaMemcpyAsync(fm->adaScal, sc, 16, cudaMemcpyHostToDevice, ctx->stream));
  }
  CK(cudaMemsetAsync(fm->dG, 0, (size_t)(2 * nP + 2 * d + dd + 8) * 8, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  fm->adaReady = true;
  return NIMFM_OK;
}

int32_t nimfm_fm_adagrad_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_adagrad_cfg *cfg,
                               int64_t *it, const int64_t *perm, int64_t nRows, double *viol, double *lossSum) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int rc = check_fm_ds(ctx, fm, X, true);
  if (rc) return rc;
  REQUIRE(cfg && it, "NULL argument");
  if (!fm->adaReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_fm_adagrad_init was not called");
  REQUIRE(cfg->miniBatchSize >= 1, "miniBatchSize < 1");
  REQUIRE(nRows >= 0 && (perm != nullptr || nRows <= X->n), "bad nRows");
  const int64_t nP = fm->nP(), d = fm->d, dd = fm->dd();
  const int32_t *idxDev = nullptr;
  if (perm && nRows > 0) {
    if ((rc = nimfm_stage_row_ids(ctx, perm, nRows, X->n))) return rc;
    idxDev = ctx->idx32Scratch;
  }
  CK(cudaMemsetAsync(ctx->scalars, 0, 16, ctx->stream));
  double *dGsP = fm->dG, *dGnP = fm->dG + nP, *dGsw = fm->dG + 2 * nP, *dGnw = fm->dG + 2 * nP + d;
  // delta block: [dGsP | dGnP | dGsw | dGnw | loss, sum dL, sum dL^2, - ] (one all-reduce), then the
  // per-feature row counts of the batch (their own small all-reduce) and the refresh pass's viol
  double *part = fm->dG + 2 * nP + 2 * d;
  double *cntF = part + 4;
  double *violPart = cntF + dd;
  const int64_t nDelta = 2 * nP + 2 * d + 4;
  const int64_t mb = cfg->miniBatchSize;
  const int SB8 = fm->nOrders * fm->k;
  // miniBatchSize = 1 on one rank: the reference's per-sample loop in one persistent block (adagrad_seq.cuh)
  {
    const int zmax = (int)std::max<int64_t>(X->maxSegNnz + fm->nAug, 1);
    const size_t smem = (3 * (size_t)zmax * SB8 + 2 * (size_t)zmax) * 8 + (size_t)zmax * 8;
    const char *env = getenv("NIMFM_ADAGRAD_SEQ");
    if (mb == 1 && ctx->nranks == 1 && nRows > 0 && SB8 <= ADASEQ_THREADS && smem + 2048 <= (size_t)ctx->smemOptin &&
        !(env && env[0] == '0')) {
      // degree 1 (SB8 = 0) takes the staged kernel: its P passes are empty loops, while the pipelined kernel
      // divides by SB8
      AdaSeqArgs q;
      memset(&q, 0, sizeof(q));
      q.data = X->data; q.indices = X->indices; q.indptr = X->indptr; q.y = X->y; q.perm = idxDev;
      q.nRows = nRows; q.d = d;
      q.degree = fm->degree; q.k = fm->k; q.nOrders = fm->nOrders; q.nAug = fm->nAug;
      q.fitLinear = fm->fitLinear; q.fitIntercept = fm->fitIntercept;
      q.P = fm->P; q.gsP = fm->gsP; q.gnP = fm->gnP; q.w = fm->w; q.gsw = fm->gsw; q.gnw = fm->gnw;
      q.b = fm->b; q.adaScal = fm->adaScal; q.scal = ctx->scalars;
      q.loss = cfg->loss; q.thr = cfg->huberThreshold;
      q.eta0 = cfg->eta0; q.alpha0 = cfg->alpha0; q.alpha = cfg->alpha; q.beta = cfg->beta;
      q.it0 = *it; q.zmax = zmax;
      const size_t smemPipe = (3 * (size_t)zmax * SB8 + (size_t)SB8 * (NIMFM_MAX_DEGREE + 1) + 3 * (size_t)zmax) * 8 +
                              2 * (size_t)zmax * 4 + (size_t)SB8 + 16;
      if (SB8 > 0 && zmax <= 64 && smemPipe + 4096 <= (size_t)ctx->smemOptin && !(env && env[0] == 's')) {   // NIMFM_ADAGRAD_SEQ=staged
        CK(cudaFuncSetAttribute(adagrad_fm_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemPipe));
        adagrad_fm_pipe_kernel<<<1, ADAPIPE_THREADS, smemPipe, ctx->stream>>>(q);
      } else {
        CK(cudaFuncSetAttribute(adagrad_fm_seq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        adagrad_fm_seq_kernel<<<1, ADASEQ_THREADS, smem, ctx->stream>>>(q);
      }
      LAUNCHED(ctx);
      CK(cudaGetLastError());
      CK(cudaMemcpyAsync(ctx->hostScalars, ctx->scalars, 16, cudaMemcpyDeviceToHost, ctx->stream));
      CK(cudaStreamSynchronize(ctx->stream));
      *it += nRows;
      if (lossSum) *lossSum = ctx->hostScalars[0];
      if (viol) *viol = ctx->hostScalars[1];
      return NIMFM_OK;
    }
  }
  MbSchedule sch;
  if ((rc = nimfm_mb_schedule(ctx, nRows, mb, *it, &sch))) return rc;
  PeerScope peers(ctx, {fm->dG});
  if (peers.rc) return peers.rc;
  // NIMFM_DETERMINISTIC=1 with miniBatchSize > 1: the gradient sums and their squares come from the column route
  // (fm_cols.cu) over the minibatch's own column index (nimfm_mb_index_build), added in sample order without atomics.
  // A one-row minibatch adds each element once (a CSR row holds a feature once): the RED route is already
  // reproducible there and keeps it.
  const char *envDet = getenv("NIMFM_DETERMINISTIC");
  const bool det = envDet && envDet[0] == '1' && mb > 1;
  TraceReport traceReport{ctx, "deterministic adagrad epoch", det};
  for (int64_t t = 0; t < sch.T; t++) {
    const int64_t start = std::min(t * mb, nRows);
    const int64_t cnt = sch.local(t);   // 0 once this rank's (shorter) shard is used up: it still joins the collectives
    const int32_t *rows = idxDev ? idxDev + start : nullptr;
    const double tIt = (double)(*it - 1);
    const int first = (*it == 1);
    {
      // per-feature row counts of the batch (all ranks): they weight viol in the refresh pass and tell
      // the refresh / apply passes which features the batch touches
      const int cgrid = (int)std::min<int64_t>((cnt * 32 + 255) / 256, (int64_t)ctx->numSMs * 16);
      adagrad_count_kernel<<<cgrid < 1 ? 1 : cgrid, 256, 0, ctx->stream>>>(X->indices, X->indptr, X->n, start, cnt, rows,
                                                                          d, fm->nAug, cntF, X->hotSlot, X->hotList, X->nHot);
      LAUNCHED(ctx);
      if ((rc = nimfm_allreduce_sum(ctx, cntF, dd))) return rc;
    }
    if (!first) {
      // update() (adagrad.nim:87-110), once per touched feature
      const int rgrid = ew_grid(ctx, std::max(nP, dd));
      if ((rc = nimfm_ensure_partials(ctx, (size_t)rgrid * 4))) return rc;
      adagrad_refresh_kernel<<<rgrid, 256, 0, ctx->stream>>>(fm->P, fm->gsP, fm->gnP, dd, SB8, cntF, fm->w, fm->gsw,
                                                             fm->gnw, d, fm->fitLinear, cfg->eta0, tIt, cfg->alpha,
                                                             cfg->beta, ctx->partials);
      LAUNCHED(ctx);
      reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(ctx->partials, rgrid, violPart, 0);
      LAUNCHED(ctx);
    }
    // one rank: the gradients and their squares go straight into g_sum / g_norm (nothing reads them before
    // the next minibatch's refresh), so the delta block and the apply pass are only needed for the all-reduce
    const bool direct = ctx->nranks == 1;
    if (det) {
      nimfm_trace_begin(ctx, "det index");
      nimfm_mb_index *ix = nullptr;
      rc = nimfm_mb_index_build(ctx, X, fm->nAug, start, cnt, rows, &ix);
      nimfm_trace_end(ctx);
      if (rc) return rc;
      nimfm_trace_begin(ctx, "det passes");
      // the intercept every row of the minibatch sees (the row kernels' AdaGrad prologue, fm_rows.cuh)
      adagrad_bias_kernel<<<1, 1, 0, ctx->stream>>>(ix->bias, fm->b, fm->adaScal, fm->fitIntercept, first, cfg->eta0,
                                                    tIt, cfg->alpha0);
      LAUNCHED(ctx);
      RowPlan pl;
      if ((rc = plan_rows(ctx, fm, &ix->view, cnt, MODE_STASH, &pl))) return rc;
      RowArgs base;
      fill_row_args(base, fm, &ix->view);
      base.b = ix->bias;
      FmDetTargets o;
      o.gP = direct ? fm->gsP : dGsP;
      o.gw = direct ? fm->gsw : dGsw;
      o.gnP = direct ? fm->gnP : dGnP;
      o.gnw = direct ? fm->gnw : dGnw;
      o.red4 = part;
      o.yhat = ix->yhat;
      rc = nimfm_fm_det_pass(ctx, fm, &ix->tw, pl, cfg->loss, cfg->huberThreshold, 0, cnt, 1.0, nullptr, base, o);
      nimfm_trace_end(ctx);
      if (rc) return rc;
    } else {
      RowPlan pl;
      if ((rc = plan_rows(ctx, fm, X, cnt, MODE_ADAGRAD, &pl))) return rc;
      RowKernel kern = pl.kern;
      if ((rc = nimfm_ensure_partials(ctx, (size_t)pl.nWarps * 4))) return rc;
      RowArgs a;
      fill_row_args(a, fm, X);
      a.rowBegin = start;
      a.nRows = cnt;
      a.rowIdx = rows;
      a.gP = direct ? fm->gsP : dGsP;
      a.gw = direct ? fm->gsw : dGsw;
      a.dGnP = direct ? fm->gnP : dGnP;
      a.dGnw = direct ? fm->gnw : dGnw;
      a.partials = ctx->partials;
      a.loss = cfg->loss;
      a.thr = cfg->huberThreshold;
      a.gsP = fm->gsP; a.gnP = fm->gnP; a.gsw = fm->gsw; a.gnw = fm->gnw; a.adaScal = fm->adaScal;
      a.eta0 = cfg->eta0; a.tIt = tIt; a.alpha0 = cfg->alpha0; a.alpha = cfg->alpha; a.beta = cfg->beta;
      a.first = first;
      a.G = pl.G;
      a.CH = pl.CH;
      kern<<<pl.grid, pl.block, pl.smem, ctx->stream>>>(a);
      LAUNCHED(ctx);
      reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(ctx->partials, pl.nWarps, part, 0);
      LAUNCHED(ctx);
    }
    // synchronous data parallelism: all-reduce the deltas [dGs | dGn | dGsw | dGnw | loss, dL, dL^2, -]
    if ((rc = nimfm_allreduce_sum(ctx, fm->dG, nDelta))) return rc;
    adagrad_scalar_kernel<<<1, 1, 0, ctx->stream>>>(fm->b, fm->adaScal, part, violPart, ctx->scalars, fm->fitIntercept,
                                                    cfg->eta0, tIt, cfg->alpha0, first);
    LAUNCHED(ctx);
    if (direct) {
      CK(cudaMemsetAsync(cntF, 0, (size_t)dd * 8, ctx->stream));
    } else {
      adagrad_apply_kernel<<<ew_grid(ctx, std::max(nP, dd)), 256, 0, ctx->stream>>>(fm->gsP, fm->gnP, dGsP, dGnP, nP, fm->gsw, fm->gnw,
                                                                     dGsw, dGnw, d, fm->fitLinear, cntF, dd);
      LAUNCHED(ctx);
    }
    *it += sch.global(t);
  }
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ctx->hostScalars, ctx->scalars, 16, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (lossSum) *lossSum = ctx->hostScalars[0];
  if (viol) *viol = ctx->hostScalars[1];
  return NIMFM_OK;
}

int32_t nimfm_fm_adagrad_finalize(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_adagrad_cfg *cfg, int64_t it) {
  if (!ctx || !fm || !cfg) return NIMFM_ERR_INVALID;
  if (!fm->adaReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_fm_adagrad_init was not called");
  CK(cudaSetDevice(ctx->device));
  adagrad_finalize_kernel<<<ew_grid(ctx, std::max(fm->nP(), fm->d)), 256, 0, ctx->stream>>>(
      fm->P, fm->gsP, fm->gnP, fm->nP(), fm->w, fm->gsw, fm->gnw, fm->d, fm->fitLinear, fm->b, fm->adaScal,
      fm->fitIntercept, cfg->eta0, (double)(it - 1), cfg->alpha0, cfg->alpha, cfg->beta);
  LAUNCHED(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  return NIMFM_OK;
}

static int permute_solver(nimfm_ctx *ctx, nimfm_fm *fm, double *hostSolver, double *dev, int toDev) {
  const int64_t nP = fm->nP();
  if (nP == 0) return NIMFM_OK;   // degree 1: no P
  double *tmp = nullptr;
  CK(cudaMalloc(&tmp, (size_t)nP * 8));
  if (toDev) CK(cudaMemcpyAsync(tmp, hostSolver, (size_t)nP * 8, cudaMemcpyHostToDevice, ctx->stream));
  permute_solver_dev<<<ew_grid(ctx, nP), 256, 0, ctx->stream>>>(tmp, dev, fm->nOrders, fm->k, fm->dd(), toDev);
  LAUNCHED(ctx);
  if (!toDev) CK(cudaMemcpyAsync(hostSolver, tmp, (size_t)nP * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaFree(tmp));
  CK(cudaGetLastError());
  return NIMFM_OK;
}

int32_t nimfm_fm_adagrad_get_state(nimfm_ctx *ctx, nimfm_fm *fm, double *gsP, double *gnP, double *gsw, double *gnw,
                                   double *gsb, double *gnb) {
  if (!ctx || !fm) return NIMFM_ERR_INVALID;
  if (!fm->adaReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_fm_adagrad_init was not called");
  CK(cudaSetDevice(ctx->device));
  int rc;
  if (gsP && (rc = permute_solver(ctx, fm, gsP, fm->gsP, 0))) return rc;
  if (gnP && (rc = permute_solver(ctx, fm, gnP, fm->gnP, 0))) return rc;
  if (gsw) CK(cudaMemcpy(gsw, fm->gsw, (size_t)fm->d * 8, cudaMemcpyDeviceToHost));
  if (gnw) CK(cudaMemcpy(gnw, fm->gnw, (size_t)fm->d * 8, cudaMemcpyDeviceToHost));
  double sc[2];
  CK(cudaMemcpy(sc, fm->adaScal, 16, cudaMemcpyDeviceToHost));
  if (gsb) *gsb = sc[0];
  if (gnb) *gnb = sc[1];
  return NIMFM_OK;
}

int32_t nimfm_fm_adagrad_set_state(nimfm_ctx *ctx, nimfm_fm *fm, const double *gsP, const double *gnP,
                                   const double *gsw, const double *gnw, double gsb, double gnb) {
  if (!ctx || !fm) return NIMFM_ERR_INVALID;
  if (!fm->adaReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_fm_adagrad_init was not called");
  REQUIRE(((gsP && gnP) || fm->nP() == 0) && gsw && gnw, "NULL state array");
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = permute_solver(ctx, fm, const_cast<double *>(gsP), fm->gsP, 1))) return rc;
  if ((rc = permute_solver(ctx, fm, const_cast<double *>(gnP), fm->gnP, 1))) return rc;
  CK(cudaMemcpy(fm->gsw, gsw, (size_t)fm->d * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(fm->gnw, gnw, (size_t)fm->d * 8, cudaMemcpyHostToDevice));
  const double sc[2] = {gsb, gnb};
  CK(cudaMemcpy(fm->adaScal, sc, 16, cudaMemcpyHostToDevice));
  return NIMFM_OK;
}

}  // extern "C"

// ================================================================== K2 fed from host buffers (end-to-end path)
__global__ void narrow_rebase_kernel(const int64_t *idx64, int32_t *idx32, int64_t nnz, int64_t *indptr,
                                     int64_t nRowsPlus1, int64_t base, int64_t d, int *bad) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  for (int64_t q = tid; q < nnz; q += stride) {
    int64_t v = idx64[q];
    if (v < 0 || v >= d) { *bad = 1; v = 0; }
    idx32[q] = (int32_t)v;
  }
  for (int64_t r = tid; r < nRowsPlus1; r += stride) indptr[r] -= base;
}


struct HotLists { int32_t v[32]; };   // [0,16): entries to clear, [16,32): entries to set (-1 = none)
static __global__ void set_hot_table_kernel(uint8_t *slot, const HotLists hl) {
  const int t = threadIdx.x;
  if (t < 16 && hl.v[t] >= 0) slot[hl.v[t]] = 255;
  __syncthreads();
  if (t >= 16 && hl.v[t] >= 0) slot[hl.v[t]] = (uint8_t)(t - 16);
}

static int ensure_stage(nimfm_ctx *ctx, nimfm_ctx::Stage &st, size_t rows, size_t nnz, bool needIdx64) {
  if (st.capRows < rows) {
    if (st.y) CK(cudaFree(st.y));
    if (st.indptr) CK(cudaFree(st.indptr));
    CK(cudaMalloc(&st.y, rows * 8));
    CK(cudaMalloc(&st.indptr, (rows + 1) * 8));
    st.capRows = rows;
  }
  if (st.capNnz < nnz) {
    if (st.data) CK(cudaFree(st.data));
    if (st.idx32) CK(cudaFree(st.idx32));
    CK(cudaMalloc(&st.data, nnz * 8));
    CK(cudaMalloc(&st.idx32, nnz * 4));
    st.capNnz = nnz;
  }
  if (needIdx64 && st.capIdx64 < nnz) {   // only the device-narrowing path stages 64-bit ids
    if (st.idx64) CK(cudaFree(st.idx64));
    st.idx64 = nullptr;
    st.capIdx64 = 0;
    CK(cudaMalloc(&st.idx64, nnz * 8));
    st.capIdx64 = nnz;
  }
  return NIMFM_OK;
}

// pinned host slots of the staging team (host_stage.h): int32 ids + rebased indptr, kSlots deep
static int ensure_host_slots(nimfm_ctx *ctx, size_t rows, size_t nnz) {
  // a capacity is only recorded once ALL slots have it: a failed allocation half way leaves it at 0, so the
  // next call reallocates every slot instead of copying from a null one
  const bool growNnz = ctx->hostCapNnz < nnz, growRows = ctx->hostCapRows < rows;
  if (growNnz) ctx->hostCapNnz = 0;
  if (growRows) ctx->hostCapRows = 0;
  for (int s = 0; s < HostStageTeam::kSlots; s++) {
    if (growNnz) {
      if (ctx->hostIdx[s]) CK(cudaFreeHost(ctx->hostIdx[s]));
      ctx->hostIdx[s] = nullptr;
      CK(cudaHostAlloc(&ctx->hostIdx[s], nnz * 4, cudaHostAllocDefault));
    }
    if (growRows) {
      if (ctx->hostPtr[s]) CK(cudaFreeHost(ctx->hostPtr[s]));
      ctx->hostPtr[s] = nullptr;
      CK(cudaHostAlloc(&ctx->hostPtr[s], (rows + 1) * 8, cudaHostAllocDefault));
    }
    if (!ctx->evSlot[s]) CK(cudaEventCreateWithFlags(&ctx->evSlot[s], cudaEventDisableTiming));
  }
  if (growNnz) ctx->hostCapNnz = nnz;
  if (growRows) ctx->hostCapRows = rows;
  return NIMFM_OK;
}

// pinned value / target slots for PAGEABLE callers (same all-or-nothing capacity rule)
static int ensure_host_value_slots(nimfm_ctx *ctx, size_t rows, size_t nnz) {
  const bool growD = ctx->hostCapData < nnz, growY = ctx->hostCapY < rows;
  if (growD) ctx->hostCapData = 0;
  if (growY) ctx->hostCapY = 0;
  for (int s = 0; s < HostStageTeam::kSlots; s++) {
    if (growD) {
      if (ctx->hostData[s]) CK(cudaFreeHost(ctx->hostData[s]));
      ctx->hostData[s] = nullptr;
      CK(cudaHostAlloc(&ctx->hostData[s], nnz * 8, cudaHostAllocDefault));
    }
    if (growY) {
      if (ctx->hostY[s]) CK(cudaFreeHost(ctx->hostY[s]));
      ctx->hostY[s] = nullptr;
      CK(cudaHostAlloc(&ctx->hostY[s], (rows + 1) * 8, cudaHostAllocDefault));
    }
  }
  if (growD) ctx->hostCapData = nnz;
  if (growY) ctx->hostCapY = rows;
  return NIMFM_OK;
}

// pinned slots + device buffers of the packed value transport (host_stage.h, pack_values)
static int ensure_pack_buffers(nimfm_ctx *ctx, size_t nnz) {
  const size_t words = nnz / 64 + 8, blks = nnz / 256 + 8;
  if (ctx->hostCapPack < nnz) {
    ctx->hostCapPack = 0;
    for (int s = 0; s < HostStageTeam::kSlots; s++) {
      if (ctx->hostPack[s]) CK(cudaFreeHost(ctx->hostPack[s]));
      if (ctx->hostMask[s]) CK(cudaFreeHost(ctx->hostMask[s]));
      if (ctx->hostBlk[s]) CK(cudaFreeHost(ctx->hostBlk[s]));
      ctx->hostPack[s] = nullptr; ctx->hostMask[s] = nullptr; ctx->hostBlk[s] = nullptr;
      CK(cudaHostAlloc(&ctx->hostPack[s], (nnz + 8) * 8, cudaHostAllocDefault));
      CK(cudaHostAlloc(&ctx->hostMask[s], words * 8, cudaHostAllocDefault));
      CK(cudaHostAlloc(&ctx->hostBlk[s], blks * 4, cudaHostAllocDefault));
    }
    ctx->hostCapPack = nnz;
  }
  for (int s = 0; s < 2; s++) {
    nimfm_ctx::Stage &st = ctx->stage[s];
    if (st.capPack < nnz) {
      if (st.packed) CK(cudaFree(st.packed));
      if (st.mask) CK(cudaFree(st.mask));
      if (st.blk) CK(cudaFree(st.blk));
      st.packed = nullptr; st.mask = nullptr; st.blk = nullptr; st.capPack = 0;
      CK(cudaMalloc(&st.packed, (nnz + 8) * 8));
      CK(cudaMalloc(&st.mask, words * 8));
      CK(cudaMalloc(&st.blk, blks * 4));
      st.capPack = nnz;
    }
  }
  return NIMFM_OK;
}

// values back from their packed transport: bit q of mask = "value q is exactly 1.0"; the others sit in `packed`,
// blk[q / 256] = index of the first packed value of q's block of 256 nonzeros
__global__ void expand_values_kernel(const uint64_t *__restrict__ mask, const uint32_t *__restrict__ blk,
                                     const double *__restrict__ packed, double *__restrict__ out, int64_t nnz) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nnz; q += stride) {
    const int64_t w = q >> 6;
    const int bit = (int)(q & 63);
    const uint64_t word = mask[w];
    if ((word >> bit) & 1) {
      out[q] = 1.0;
    } else {
      uint32_t idx = blk[q >> 8];
      for (int64_t v = (q >> 8) << 2; v < w; v++) idx += __popcll(~mask[v]);
      idx += __popcll(~word & ((1ull << bit) - 1ull));
      out[q] = packed[idx];
    }
  }
}

// is this host pointer outside every page-locked allocation CUDA knows (a plain malloc / Nim seq / numpy array)?
static bool is_pageable(const void *p) {
  if (!p) return false;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return at.type == cudaMemoryTypeUnregistered;
}

// Rows [0,nRows) of a HOST CSR streamed through the row kernel in chunks, the H2D copy of chunk c+1
// overlapping the kernel of chunk c.  predOut == NULL: predict+grad (K2) into the model's gradient
// buffers; predOut != NULL: decisionFunction (K1), each chunk's predictions copied back as it finishes.
static int stream_host_rows(nimfm_ctx *ctx, nimfm_fm *fm, int64_t nRows, int64_t d, const double *data,
                            const int64_t *indices, const int64_t *indptr, const double *y, int32_t loss,
                            double huberThreshold, int64_t miniBatchSize, int64_t chunkRows, int32_t zeroGrads,
                            int32_t allreduce, double *lossSum, double *predOut) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  const bool predict = predOut != nullptr;
  REQUIRE(fm && indptr && (y || predict), "NULL argument");
  REQUIRE(d == fm->d, "Invalid nFeatures. (batch %lld, model %lld)", (long long)d, (long long)fm->d);
  REQUIRE(nRows >= 0 && miniBatchSize >= 1, "bad nRows / miniBatchSize");
  if (chunkRows <= 0) chunkRows = 1 << 17;   // 84 MB per chunk at 39 nnz/row: short pipeline ramp and tail
  const int64_t nG = fm->nP() + fm->d + 2;
  PeerScope peers(ctx, {(!predict && allreduce) ? fm->grad : nullptr});
  if (peers.rc) return peers.rc;
  if (zeroGrads && !predict) CK(cudaMemsetAsync(fm->grad, 0, (size_t)nG * 8, ctx->stream));
  int *bad = reinterpret_cast<int *>(ctx->scalars + 60);
  CK(cudaMemsetAsync(bad, 0, sizeof(int), ctx->stream));
  // the chunk list; the two device staging sets are sized for the largest chunk
  std::vector<HostChunk> chunks;
  size_t maxNnz = 1;
  for (int64_t r0 = 0; r0 < nRows; r0 += chunkRows) {
    HostChunk ch;
    ch.r0 = r0;
    ch.r1 = std::min(nRows, r0 + chunkRows);
    REQUIRE(indptr[ch.r1] >= indptr[ch.r0], "indptr is not monotone");
    ch.base = indptr[ch.r0];
    ch.nnz = indptr[ch.r1] - ch.base;
    maxNnz = std::max(maxNnz, (size_t)ch.nnz);
    chunks.push_back(ch);
  }
  const int64_t nChunks = (int64_t)chunks.size();
  // host staging (host_stage.h): ids narrowed to int32 and indptr rebased by a thread team into pinned slots,
  // 12 instead of 16 bytes per nonzero on the link; small calls and thread-starved ranks narrow on the device
  const int64_t stageMinNnz = getenv("NIMFM_HOST_STAGE_MIN_NNZ") ? atoll(getenv("NIMFM_HOST_STAGE_MIN_NNZ")) : (1 << 20);
  const bool bigCall = indices && nRows > 0 && indptr[nRows] - indptr[0] >= stageMinNnz;
  // packed transport of the values when at least a quarter of a sample of them is exactly 1.0 (one-hot data) AND the
  // rank has the host threads for it: lossless, 281 instead of 484 bytes per Criteo-shaped row on the link, but the
  // team then reads the values too and becomes the bound -- measured on this box's 16 cores: 8 threads 83 M rows/s
  // (worse than the 107 M of the raw route, which is link-bound), 14 threads 127 M (host-memory-bound).
  // NIMFM_HOST_PACK=0 / 1 forces it off / on.
  bool packValues = false;
  if (bigCall && data && HostStageTeam::pageable_threads(ctx->nranks) >= 12) {
    const int64_t nnzAll = indptr[nRows] - indptr[0], sample = std::min<int64_t>(nnzAll, 1 << 16);
    int64_t ones = 0;
    for (int64_t q = 0; q < sample; q++) ones += data[indptr[0] + q * (nnzAll / sample)] == 1.0;
    packValues = ones * 4 >= sample;
  }
  if (const char *e = getenv("NIMFM_HOST_PACK")) packValues = bigCall && data && e[0] == '1';
  const int hostT = !bigCall ? 0 : ((packValues || is_pageable(data)) ? HostStageTeam::pageable_threads(ctx->nranks)
                                                                       : HostStageTeam::default_threads(ctx->nranks));
  if (hostT == 0) packValues = false;
  int rc;
  const size_t capRows = (size_t)std::min(nRows, chunkRows) + 1;
  for (int s = 0; s < 2; s++)
    if ((rc = ensure_stage(ctx, ctx->stage[s], capRows, maxNnz, hostT == 0))) return rc;
  if (hostT > 0 && (rc = ensure_host_slots(ctx, capRows, maxNnz))) return rc;
  if (!ctx->stageHotSlot || ctx->stageHotD != d) {   // persistent hot-column table, all cold
    if (ctx->stageHotSlot) CK(cudaFree(ctx->stageHotSlot));
    ctx->stageHotSlot = nullptr;
    CK(cudaMalloc(&ctx->stageHotSlot, (size_t)std::max<int64_t>(d, 1)));
    CK(cudaMemsetAsync(ctx->stageHotSlot, 255, (size_t)std::max<int64_t>(d, 1), ctx->stream));
    if (!ctx->stageHotList) CK(cudaMalloc(&ctx->stageHotList, 32 * sizeof(int32_t)));
    ctx->stageHotD = d;
    ctx->stageNHot = 0;
  }
  std::unique_ptr<HostStageTeam> team;
  // pageable caller arrays: their values (and targets) travel through the team's pinned slots as well
  const bool pageable = hostT > 0 && is_pageable(data);
  const bool stageValues = pageable && !packValues;
  if ((pageable || packValues) && (rc = ensure_host_value_slots(ctx, capRows, packValues ? 1 : maxNnz))) return rc;
  if (packValues && (rc = ensure_pack_buffers(ctx, maxNnz))) return rc;
  if (hostT > 0) {
    team.reset(new HostStageTeam(hostT, indices, indptr, d, chunks, ctx->hostIdx, ctx->hostPtr));
    if (packValues)
      team->pack_values(data, (pageable && !predict) ? y : nullptr, ctx->hostPack, ctx->hostMask, ctx->hostBlk, ctx->hostY);
    else if (stageValues)
      team->stage_values(data, predict ? nullptr : y, ctx->hostData, ctx->hostY);
    team->allow(std::min<int64_t>(nChunks, HostStageTeam::kSlots - 1));
  }
  const bool stageY = pageable;
  // a failed check leaves with both streams drained (copies read the caller's buffers and our pinned slots)
  auto drained = [&](int code) {
    cudaStreamSynchronize(ctx->copyStream);
    cudaStreamSynchronize(ctx->stream);
    return code;
  };
  int nHot = 0;
  int64_t h2d = 0, d2h = 0;
  double *dOutAll = nullptr;
  if (predict && nRows > 0 && is_pageable(predOut)) CK(cudaMalloc(&dOutAll, (size_t)nRows * 8));
  struct OutGuard {
    double *&p;
    ~OutGuard() { if (p) cudaFree(p); }
  } outGuard{dOutAll};
  for (int64_t c = 0; c < nChunks; c++) {
    const int64_t r0 = chunks[c].r0, r1 = chunks[c].r1, rows = r1 - r0;
    const int64_t base = chunks[c].base, nnz = chunks[c].nnz;
    nimfm_ctx::Stage &st = ctx->stage[c & 1];
    const int hs = (int)(c % HostStageTeam::kSlots);
    HostChunkInfo info;
    if (team) {
      info = team->wait(c);   // normally already staged: the team runs two chunks ahead of the copies
      if (info.minSeg < 0)
        return drained(nimfm_fail(ctx, NIMFM_ERR_INVALID, "indptr is not monotone in rows [%lld,%lld)", (long long)r0, (long long)r1));
      if (info.bad)
        return drained(nimfm_fail(ctx, NIMFM_ERR_INVALID, "column index out of range [0,%lld)", (long long)d));
    }
    // the copies go out first; the host-side bookkeeping below overlaps with the DMA
    if (c >= 2) CK(cudaStreamWaitEvent(ctx->copyStream, ctx->evComputed[c & 1], 0));   // buffer is free again
    int64_t valueBytes = nnz * 8;
    if (packValues) {
      const int64_t per = team->slice_len(nnz);
      valueBytes = 0;
      for (int t = 0; t < team->threads(); t++) {
        const int64_t a0 = std::min(nnz, per * t), cnt = info.packed[t];
        if (cnt > 0)
          CK(cudaMemcpyAsync(st.packed + a0, ctx->hostPack[hs] + a0, (size_t)cnt * 8, cudaMemcpyHostToDevice, ctx->copyStream));
        valueBytes += cnt * 8;
      }
      const int64_t words = (nnz + 63) / 64, blks = (nnz + 255) / 256;
      if (nnz > 0) {
        CK(cudaMemcpyAsync(st.mask, ctx->hostMask[hs], (size_t)words * 8, cudaMemcpyHostToDevice, ctx->copyStream));
        CK(cudaMemcpyAsync(st.blk, ctx->hostBlk[hs], (size_t)blks * 4, cudaMemcpyHostToDevice, ctx->copyStream));
      }
      valueBytes += words * 8 + blks * 4;
    } else {
      CK(cudaMemcpyAsync(st.data, stageValues ? ctx->hostData[hs] : data + base, (size_t)nnz * 8, cudaMemcpyHostToDevice,
                         ctx->copyStream));
    }
    if (team) {
      CK(cudaMemcpyAsync(st.idx32, ctx->hostIdx[hs], (size_t)nnz * 4, cudaMemcpyHostToDevice, ctx->copyStream));
      CK(cudaMemcpyAsync(st.indptr, ctx->hostPtr[hs], (size_t)(rows + 1) * 8, cudaMemcpyHostToDevice, ctx->copyStream));
    } else {
      CK(cudaMemcpyAsync(st.idx64, indices + base, (size_t)nnz * 8, cudaMemcpyHostToDevice, ctx->copyStream));
      CK(cudaMemcpyAsync(st.indptr, indptr + r0, (size_t)(rows + 1) * 8, cudaMemcpyHostToDevice, ctx->copyStream));
    }
    if (!predict)
      CK(cudaMemcpyAsync(st.y, stageY ? ctx->hostY[hs] : y + r0, (size_t)rows * 8, cudaMemcpyHostToDevice, ctx->copyStream));
    CK(cudaEventRecord(ctx->evCopied[c & 1], ctx->copyStream));
    if (team) CK(cudaEventRecord(ctx->evSlot[hs], ctx->copyStream));
    h2d += valueBytes + nnz * (team ? 4 : 8) + (rows + 1) * 8 + (predict ? 0 : rows * 8);
    d2h += predict ? rows * 8 : 0;
    if (c == 0 && !predict) {
      // hot columns of this batch (row sample on the host; see nimfm_find_hot): the previous call's
      // entries are cleared and the new ones set by one tiny kernel on the persistent table
      std::vector<int32_t> hot;
      nHot = (indices && nRows > 0) ? nimfm_find_hot(indices, indptr, 0, nRows, hot, 2048, d) : 0;
      int32_t lists[32];
      for (int i = 0; i < 16; i++) lists[i] = i < ctx->stageNHot ? ctx->stagePrevHot[i] : -1;
      for (int i = 0; i < 16; i++) lists[16 + i] = i < nHot ? hot[i] : -1;
      CK(cudaMemcpyAsync(ctx->stageHotList, lists + 16, 16 * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
      HotLists hl;
      memcpy(hl.v, lists, sizeof(lists));
      set_hot_table_kernel<<<1, 32, 0, ctx->stream>>>(ctx->stageHotSlot, hl);
      LAUNCHED(ctx);
      for (int i = 0; i < nHot; i++) ctx->stagePrevHot[i] = hot[i];
      ctx->stageNHot = nHot;
    }
    if (!team) {
      for (int64_t r = r0; r < r1; r++) {
        const int64_t len = indptr[r + 1] - indptr[r];
        info.maxSeg = std::max(info.maxSeg, len);
        info.minSeg = std::min(info.minSeg, len);
      }
      if (info.minSeg < 0)
        return drained(nimfm_fail(ctx, NIMFM_ERR_INVALID, "indptr is not monotone in rows [%lld,%lld)", (long long)r0, (long long)r1));
    }
    CK(cudaStreamWaitEvent(ctx->stream, ctx->evCopied[c & 1], 0));
    if (packValues && nnz > 0) {
      expand_values_kernel<<<ew_grid(ctx, nnz), 256, 0, ctx->stream>>>(st.mask, st.blk, st.packed, st.data, nnz);
      LAUNCHED(ctx);
    }
    if (!team) {
      narrow_rebase_kernel<<<ew_grid(ctx, nnz), 256, 0, ctx->stream>>>(st.idx64, st.idx32, nnz, st.indptr, rows + 1,
                                                                       base, d, bad);
      LAUNCHED(ctx);
    }
    nimfm_dataset tmp;
    tmp.kind = NIMFM_DS_CSR;
    tmp.n = rows;
    tmp.d = d;
    tmp.nnz = nnz;
    tmp.maxSegNnz = info.maxSeg;
    tmp.data = st.data;
    tmp.indices = st.idx32;
    tmp.indptr = st.indptr;
    tmp.y = st.y;
    tmp.hotSlot = ctx->stageHotSlot;
    tmp.hotList = ctx->stageHotList;
    tmp.nHot = nHot;
    if (predict && dOutAll) {
      // pageable result array: a device->pageable copy blocks the host until the kernel is done and would
      // serialise the pipeline, so the chunks' predictions collect on the device and leave in one staged copy
      if ((rc = nimfm_fm_predict_device_lams(ctx, fm, &tmp, dOutAll + r0))) return drained(rc);
    } else if (predict) {
      // the stage's target buffer doubles as the chunk's output; it travels back behind the kernel
      if ((rc = nimfm_fm_predict_device_lams(ctx, fm, &tmp, st.y))) return drained(rc);
      CK(cudaMemcpyAsync(predOut + r0, st.y, (size_t)rows * 8, cudaMemcpyDeviceToHost, ctx->stream));
    } else {
      if ((rc = launch_loss_grad(ctx, fm, &tmp, loss, huberThreshold, 0, rows, nullptr, (double)miniBatchSize, nullptr)))
        return drained(rc);
      add_tail_kernel<<<1, 1, 0, ctx->stream>>>(fm->grad + nG - 2, ctx->scalars + 8);
      LAUNCHED(ctx);
    }
    CK(cudaEventRecord(ctx->evComputed[c & 1], ctx->stream));
    if (team) {
      // chunk c+2 reuses the pinned slot of chunk c-2: hand it to the team once that copy has left the host
      if (c >= 2) CK(cudaEventSynchronize(ctx->evSlot[(c - 2) % HostStageTeam::kSlots]));
      team->allow(c + 3);
    }
  }
  ctx->lastH2D = h2d;
  ctx->lastD2H = d2h + (lossSum && !predict ? 8 : 0);
  ctx->lastHostThreads = hostT;
  ctx->lastPageable = pageable ? 1 : 0;
  if (!predict && allreduce && (rc = nimfm_allreduce_sum(ctx, fm->grad, nG))) return rc;
  if (dOutAll && (rc = nimfm_staged_d2h(ctx, predOut, dOutAll, (size_t)nRows * 8))) return drained(rc);
  int hbad = 0;
  CK(cudaMemcpyAsync(&hbad, bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  if (lossSum && !predict) CK(cudaMemcpyAsync(lossSum, fm->grad + nG - 1, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaStreamSynchronize(ctx->copyStream));
  CK(cudaGetLastError());
  if (hbad) return nimfm_fail(ctx, NIMFM_ERR_INVALID, "column index out of range [0,%lld)", (long long)d);
  return NIMFM_OK;
}

extern "C" int32_t nimfm_fm_loss_grad_host(nimfm_ctx *ctx, nimfm_fm *fm, int64_t nRows, int64_t d,
                                           const double *data, const int64_t *indices, const int64_t *indptr,
                                           const double *y, int32_t loss, double huberThreshold,
                                           int64_t miniBatchSize, int64_t chunkRows, int32_t zeroGrads,
                                           int32_t allreduce, double *lossSum) {
  if (ctx && !y) return nimfm_fail(ctx, NIMFM_ERR_INVALID, "y is NULL");
  return stream_host_rows(ctx, fm, nRows, d, data, indices, indptr, y, loss, huberThreshold, miniBatchSize, chunkRows,
                          zeroGrads, allreduce, lossSum, nullptr);
}

// decisionFunction (model/factorization_machine.nim:100-122) fed from HOST buffers: the serving-side twin
// of nimfm_fm_loss_grad_host (out[nRows] on the host; pinned memory gives full PCIe bandwidth)
extern "C" int32_t nimfm_fm_decision_function_host(nimfm_ctx *ctx, nimfm_fm *fm, int64_t nRows, int64_t d,
                                                   const double *data, const int64_t *indices,
                                                   const int64_t *indptr, int64_t chunkRows, double *out) {
  if (ctx && !out) return nimfm_fail(ctx, NIMFM_ERR_INVALID, "out is NULL");
  return stream_host_rows(ctx, fm, nRows, d, data, indices, indptr, nullptr, 0, 1.0, 1, chunkRows, 0, 0, nullptr, out);
}
