// sgd_mb.cu -- synchronous-minibatch SGD for FM and FFM: the deterministic device analogue of the reference's
// Hogwild variants fit(..., maxThreads) (optimizer/sgd_multi.nim:40-120, sgd_ffm_multi.nim:31-103), in which T
// lock-free threads each apply step() (sgd.nim:246-258) to parameters that are up to ~T updates stale.
//
// Here the B samples of a minibatch are all evaluated at the same parameters (one launch of the row / pair
// kernel, coef = dloss: the SUM of the per-sample gradients), then their B updates are applied at once with
// the step sizes of the minibatch's first iteration:
//     touched feature j (it occurs in the minibatch; all orders / fields of it, as update() does, :214-222):
//         p <- (1 - eta_P beta)^B p - eta_P sum_i dL_i dA_i,      viol += |p_new - p|
//     untouched feature:  p <- (1 - eta_P beta)^B p               (the lazy scaling of :231-239, applied eagerly)
//     w likewise with (eta_w, alpha); intercept b <- (1 - eta_b alpha0)^B b - eta_b sum_i dL_i
//     it += B
// With B = 1 this is step() itself (p - eta (dL dA + beta p), viol = |update|), which the tests hold against
// the sequential oracle; for B > 1 the oracle restates the rule above (oracle.sgd_minibatch_fit).
// Data parallel like MBPSGD / AdaGrad: with a communicator, X is this rank's shard, every rank feeds localBatch
// rows of each minibatch, the touch counts and the gradient buffer ([gP | gw | sum dL, loss]) are all-reduced
// and every rank applies the identical step (shards must be even: B = localBatch * ranks).
#include <algorithm>

#include "common.cuh"
#include "dense_kernels.cuh"

extern "C" {   // library-internal helpers defined inside the extern "C" blocks of fm_api.cu / ffm.cu
int nimfm_fm_launch_grad_rows(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, int loss, double thr,
                              int64_t rowBegin, int64_t nRows, const int32_t *rowIdxDev, double mb);
int nimfm_ffm_launch_grad_rows(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, int loss, double thr,
                               int64_t rowBegin, int64_t nRows, const int32_t *rowIdxDev, double mb);
double nimfm_get_eta(int sched, double eta0, double power, double reg, int64_t it);
int nimfm_fm_sgd_mb_lazy_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_sgd_cfg *cfg,
                               int64_t B, int64_t *it, const int32_t *idxDev, int64_t nRows, int *applied,
                               double *viol, double *lossSum);
}

namespace {

// (1 - eta reg)^B as B multiplications in a fixed order (the oracle does the same: bit-identical factors)
double shrink_pow(double base, int64_t B) {
  double s = 1.0;
  for (int64_t i = 0; i < B; i++) s *= base;
  return s;
}

// P rows: one thread per element.  cnt[j] > 0 marks the features of the minibatch.
__global__ void __launch_bounds__(256) sgd_mb_P_kernel(double *__restrict__ P, double *__restrict__ G, int64_t SB8,
                                                       int64_t nP, const double *__restrict__ cnt, double sP,
                                                       double negEtaP, double *violPart) {
  __shared__ double red[8];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  double viol = 0.0;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < nP; e += stride) {
    const double p = P[e];
    if (cnt[e / SB8] > 0.0) {
      const double pn = sP * p + negEtaP * G[e];
      viol += fabs(pn - p);
      P[e] = pn;
      G[e] = 0.0;
    } else {
      P[e] = sP * p;
    }
  }
  viol = block_sum(viol, red);
  if (threadIdx.x == 0) {
    violPart[blockIdx.x * 4 + 0] = viol;
    violPart[blockIdx.x * 4 + 1] = 0.0;
    violPart[blockIdx.x * 4 + 2] = 0.0;
    violPart[blockIdx.x * 4 + 3] = 0.0;
  }
}

// per-feature state: w, the touch counts (reset for the next minibatch); block 0: intercept and the loss sum.
// red4 = [loss sum, sum dL, ...] of the minibatch (reduce_partials of the row kernel's partials).
__global__ void __launch_bounds__(256) sgd_mb_feat_kernel(double *w, double *gw, int64_t d, double *cnt, int64_t dd,
                                                          double sW, double negEtaW, int fitLinear, double *b,
                                                          const double *red4, double *tail, double sB, double negEtaB,
                                                          int fitIntercept, double *scal, double *violPart) {
  __shared__ double red[8];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  double viol = 0.0;
  for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < dd; j += stride) {
    const bool touched = cnt[j] > 0.0;
    if (j < d) {
      if (fitLinear) {
        const double v = w[j];
        if (touched) {
          const double vn = sW * v + negEtaW * gw[j];
          viol += fabs(vn - v);
          w[j] = vn;
        } else {
          w[j] = sW * v;
        }
      }
      if (touched) gw[j] = 0.0;
    }
    if (touched) cnt[j] = 0.0;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    // one rank: red4 = [loss, sum dL] of the minibatch; several: the all-reduced tail [sum dL, loss] of the buffer
    const double gb = tail ? tail[0] : red4[1], ls = tail ? tail[1] : red4[0];
    if (fitIntercept) {
      const double bb = b[0], bn = sB * bb + negEtaB * gb;
      viol += fabs(bn - bb);
      b[0] = bn;
    }
    scal[0] += ls;
    if (tail) tail[0] = tail[1] = 0.0;
  }
  viol = block_sum(viol, red);
  if (threadIdx.x == 0) {
    violPart[blockIdx.x * 4 + 0] = viol;
    violPart[blockIdx.x * 4 + 1] = 0.0;
    violPart[blockIdx.x * 4 + 2] = 0.0;
    violPart[blockIdx.x * 4 + 3] = 0.0;
  }
}

struct MbModel {
  double *P, *grad, *w, *b;
  int64_t nP, SB8, d, dd;
  int nAug, fitLinear, fitIntercept;
  double **cnt;   // lazily allocated [dd] touch counts owned by the model
};

template <class LaunchGrad>
int sgd_mb_epoch(nimfm_ctx *ctx, const MbModel &M, const nimfm_dataset *X, const nimfm_sgd_cfg *cfg, int64_t B,
                 int64_t localBatch, int64_t *it, const int64_t *perm, int64_t nRows, double *viol, double *lossSum,
                 LaunchGrad launch) {
  REQUIRE(cfg && it, "NULL argument");
  REQUIRE(B >= 1, "miniBatchSize < 1");
  const int R = ctx->nranks;
  if (localBatch <= 0) localBatch = B;
  REQUIRE(R > 1 || localBatch == B, "one rank: localBatch must equal miniBatchSize");
  REQUIRE(nRows >= 0 && (perm != nullptr || nRows <= X->n), "bad nRows");
  int rc;
  const int32_t *idxDev = nullptr;
  if (perm && nRows > 0) {
    if ((rc = nimfm_stage_row_ids(ctx, perm, nRows, X->n))) return rc;
    idxDev = ctx->idx32Scratch;
  }
  if (!*M.cnt) {
    if ((rc = nimfm_comm_alloc(ctx, M.cnt, (size_t)std::max<int64_t>(M.dd, 2)))) return rc;
    CK(cudaMemsetAsync(*M.cnt, 0, (size_t)std::max<int64_t>(M.dd, 1) * 8, ctx->stream));
  }
  double *cnt = *M.cnt;
  const int64_t nG = M.nP + M.d + 2;
  CK(cudaMemsetAsync(M.grad, 0, (size_t)nG * 8, ctx->stream));
  CK(cudaMemsetAsync(ctx->scalars, 0, 8, ctx->stream));          // [0]: loss sum of the epoch
  CK(cudaMemsetAsync(ctx->scalars + 20, 0, 4 * 8, ctx->stream)); // [20]: viol of the epoch
  const int gridP = ew_grid(ctx, M.nP), gridF = ew_grid(ctx, M.dd);
  // shards and shares may be uneven: all ranks run the same number of minibatches and use the GLOBAL row count
  MbSchedule sch;
  if ((rc = nimfm_mb_schedule(ctx, nRows, localBatch, *it, &sch))) return rc;
  PeerScope peers(ctx, {M.grad, cnt});
  if (peers.rc) return peers.rc;
  TraceReport traceReport{ctx, "minibatch sgd epoch", true};   // NIMFM_TRACE=1: the deterministic index / passes spans
  for (int64_t t = 0; t < sch.T; t++) {
    const int64_t q0 = std::min(t * localBatch, nRows);
    const int64_t Bl = sch.local(t), Bm = sch.global(t);   // rows of this rank / of the whole minibatch
    const int cgrid = (int)std::max<int64_t>(1, std::min<int64_t>((Bl * 32 + 255) / 256, (int64_t)ctx->numSMs * 16));
    adagrad_count_kernel<<<cgrid, 256, 0, ctx->stream>>>(X->indices, X->indptr, X->n, q0, Bl, idxDev ? idxDev + q0 : nullptr,
                                                        M.d, M.nAug, cnt, X->hotSlot, X->hotList, X->nHot);
    LAUNCHED(ctx);
    if (Bl > 0) {
      if ((rc = launch(q0, Bl, idxDev ? idxDev + q0 : nullptr))) return rc;   // G += sum_i dL_i dA_i; red4 at scalars+8
    } else {
      CK(cudaMemsetAsync(ctx->scalars + 8, 0, 4 * 8, ctx->stream));           // this rank's shard is used up
    }
    if (R > 1) {
      add_tail_kernel<<<1, 1, 0, ctx->stream>>>(M.grad + nG - 2, ctx->scalars + 8);
      LAUNCHED(ctx);
      if ((rc = nimfm_allreduce_sum(ctx, cnt, M.dd))) return rc;
      if ((rc = nimfm_allreduce_sum(ctx, M.grad, nG))) return rc;
    }
    const double etaP = nimfm_get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->beta, *it);
    const double etaW = nimfm_get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha, *it);
    const double etaB = nimfm_get_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha0, *it);
    const double sP = shrink_pow(1.0 - etaP * cfg->beta, Bm), sW = shrink_pow(1.0 - etaW * cfg->alpha, Bm),
                 sB = shrink_pow(1.0 - etaB * cfg->alpha0, Bm);
    if ((rc = nimfm_ensure_partials(ctx, (size_t)(gridP + gridF) * 4))) return rc;
    sgd_mb_P_kernel<<<gridP, 256, 0, ctx->stream>>>(M.P, M.grad, M.SB8, M.nP, cnt, sP, -etaP, ctx->partials);
    LAUNCHED(ctx);
    sgd_mb_feat_kernel<<<gridF, 256, 0, ctx->stream>>>(M.w, M.grad + M.nP, M.d, cnt, M.dd, sW, -etaW, M.fitLinear, M.b,
                                                      ctx->scalars + 8, R > 1 ? M.grad + nG - 2 : nullptr, sB, -etaB,
                                                      M.fitIntercept, ctx->scalars, ctx->partials + (size_t)gridP * 4);
    LAUNCHED(ctx);
    reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(ctx->partials, gridP + gridF, ctx->scalars + 20, 1);
    LAUNCHED(ctx);
    *it += Bm;
  }
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ctx->hostScalars, ctx->scalars, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(ctx->hostScalars + 1, ctx->scalars + 20, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (lossSum) *lossSum = ctx->hostScalars[0];
  if (viol) *viol = ctx->hostScalars[1];
  return NIMFM_OK;
}

}  // namespace

extern "C" {

int32_t nimfm_fm_sgd_minibatch_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_sgd_cfg *cfg,
                                     int64_t miniBatchSize, int64_t localBatch, int64_t *it, const int64_t *perm,
                                     int64_t nRows, double *viol, double *lossSum) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  REQUIRE(fm && X, "NULL handle");
  REQUIRE(X->kind == NIMFM_DS_CSR || X->kind == NIMFM_DS_CSR_FIELD, "a CSR dataset is required");
  REQUIRE(X->d == fm->d, "Invalid nFeatures. (dataset %lld, model %lld)", (long long)X->d, (long long)fm->d);
  REQUIRE(X->y != nullptr, "dataset has no targets (nimfm_dataset_set_targets)");
  REQUIRE(cfg && it && miniBatchSize >= 1, "NULL argument or miniBatchSize < 1");
  REQUIRE(nRows >= 0 && (perm != nullptr || nRows <= X->n), "bad nRows");
  {
    // touched-features-only form when a minibatch touches a minority of the features (K6b over K3b)
    const int32_t *idxDev = nullptr;
    if (perm && nRows > 0) {
      int rcs = nimfm_stage_row_ids(ctx, perm, nRows, X->n);
      if (rcs) return rcs;
      idxDev = ctx->idx32Scratch;
    }
    int applied = 0;
    int rcl = nimfm_fm_sgd_mb_lazy_epoch(ctx, fm, X, cfg, miniBatchSize, it, idxDev, nRows, &applied, viol, lossSum);
    if (rcl || applied) return rcl;
  }
  MbModel M{fm->P, fm->grad, fm->w, fm->b, fm->nP(), (int64_t)fm->nOrders * fm->k, fm->d, fm->dd(), fm->nAug,
            fm->fitLinear, fm->fitIntercept, &fm->sgdCnt};
  if (fm->nOrders == 0) M.SB8 = 1;
  return sgd_mb_epoch(ctx, M, X, cfg, miniBatchSize, localBatch, it, perm, nRows, viol, lossSum,
                      [&](int64_t q0, int64_t Bm, const int32_t *idx) {
                        return nimfm_fm_launch_grad_rows(ctx, fm, X, cfg->loss, cfg->huberThreshold, q0, Bm, idx, 1.0);
                      });
}

int32_t nimfm_ffm_sgd_minibatch_epoch(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, const nimfm_sgd_cfg *cfg,
                                      int64_t miniBatchSize, int64_t localBatch, int64_t *it, const int64_t *perm,
                                      int64_t nRows, double *viol, double *lossSum) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  REQUIRE(m && X, "NULL handle");
  REQUIRE(X->kind == NIMFM_DS_CSR_FIELD, "a CSRFieldDataset is required");
  REQUIRE(X->d == m->d && X->nFields == m->nFields, "Invalid nFeatures / nFields.");
  REQUIRE(X->y != nullptr, "dataset has no targets (nimfm_dataset_set_targets)");
  MbModel M{m->P, m->grad, m->w, m->b, m->nP(), m->nFields * m->k, m->d, m->d, 0, m->fitLinear, m->fitIntercept,
            &m->sgdCnt};
  return sgd_mb_epoch(ctx, M, X, cfg, miniBatchSize, localBatch, it, perm, nRows, viol, lossSum,
                      [&](int64_t q0, int64_t Bm, const int32_t *idx) {
                        return nimfm_ffm_launch_grad_rows(ctx, m, X, cfg->loss, cfg->huberThreshold, q0, Bm, idx, 1.0);
                      });
}

}  // extern "C"
