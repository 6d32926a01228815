// cd.cu -- coordinate descent for FM / HOFM on ONE GPU (optimizer/cd.nim:29-194,
// optimizer/fit_linear.nim:5-38), SURVEY K7-K9.
//
// The coordinate loop is sequential over (order, component s, column j): update j+1 reads the
// yPred / A-cache entries update j wrote.  The parallelism that preserves the reference's results is
//   (1) inside a column: the reduction  sum_i dloss_i*dA_i , sum_i dA_i^2  and the in-place refresh
//       of A[i, 1..m], yPred[i] over the column's rows (one warp, or one block for long columns);
//   (2) across CONSECUTIVE columns whose row supports are pairwise disjoint: update j only touches
//       yPred[i], A[i,:] of its own rows (cd.nim:41-44,67-73), so such a run can be updated
//       concurrently with results identical to the sequential order.  The runs ("batches") are
//       found once per dataset (all user columns, then all item columns, for one-hot user+item data).
// One kernel launch per batch; the A-cache rebuild per component (cd.nim:58 / :85-88) is a
// row-parallel kernel over a CSR twin of the data, visiting each row's nonzeros in ascending column
// order exactly like the reference's column sweep does.
// P stays in the reference's component-major layout P[o][s][j] here (cd.fit does not transpose).
#include <math.h>
#include <stdlib.h>

#include <algorithm>

#include "dense_kernels.cuh"

int nimfm_fm_predict_device(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *Xcsr, double *dOut);

#define CD_MAXDEG NIMFM_MAX_DEGREE

struct CdState {
  nimfm_dataset *csr = nullptr;          // row-major twin (A-cache builds)
  std::vector<int64_t> batchStart;       // column batches over [0, d): batch b = [batchStart[b], batchStart[b+1])
  std::vector<int64_t> batchMaxLen;
  double *updAbs = nullptr;              // |update| of every coordinate step of one epoch (fixed-order viol sum)
  int64_t updCap = 0;
  double alpha0 = 0, alpha = 0, beta = 0;  // already multiplied by nSamples (cd.nim:123-125)
  double *chain = nullptr;                 // PCD chained prox scratch: [a | c | u] x (d + nAug)
  int64_t chainCap = 0;
  // one outer iteration is ~100-600 short kernels whose arguments do not change between iterations:
  // it is captured once into a CUDA graph and replayed (the sweep is launch-latency-bound otherwise)
  cudaGraphExec_t graph = nullptr;
  int64_t graphKernels = 0;
  struct Key {
    int prox, loss;
    double gammaRaw, thr, alpha0, alpha, beta;
  } graphKey = {0, 0, 0, 0, 0, 0, 0};
};

// cdScal layout: [0] viol, [1] loss mean, [2] reg/n, [3] sum dloss, [4] |w|^2, [5] |P|^2
static std::vector<std::pair<nimfm_fm *, CdState *>> g_cd;   // small registry: fm -> CD state

static CdState *cd_state(nimfm_fm *fm, bool create) {
  for (auto &p : g_cd)
    if (p.first == fm) return p.second;
  if (!create) return nullptr;
  g_cd.push_back({fm, new CdState()});
  return g_cd.back().second;
}

// ------------------------------------------------------------------ layout: device P[j][o][s] <-> Pcm[o][s][j]
static __global__ void cd_permute_kernel(double *D, double *R, int nO, int k, int64_t dd, int toCm) {
  const int64_t total = (int64_t)nO * k * dd;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = e % dd;
    const int64_t t = e / dd;
    const int s = (int)(t % k), o = (int)(t / k);     // e indexes Pcm
    const int64_t de = (j * nO + o) * k + s;
    if (toCm) R[e] = D[de];
    else D[de] = R[e];
  }
}

// ------------------------------------------------------------------ reductions over rows
static __global__ void cd_sum_dloss_kernel(const double *y, const double *yPred, int64_t n, int loss, double thr,
                                           double *partials) {
  __shared__ double red[8];
  double acc = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    acc += dev_dloss(loss, thr, y[i], yPred[i]);
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}
static __global__ void cd_sum_loss_kernel(const double *y, const double *yPred, int64_t n, int loss, double thr,
                                          double *partials) {
  __shared__ double red[8];
  double acc = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    acc += dev_loss(loss, thr, y[i], yPred[i]);
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}
static __global__ void cd_sumsq_kernel(const double *v, int64_t n, double *partials) {
  __shared__ double red[8];
  double acc = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    acc += v[i] * v[i];
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) partials[blockIdx.x] = acc;
}
// out[slot] = sum of partials[0..m) in a fixed order (one block)
static __global__ void cd_final_sum_kernel(const double *partials, int64_t m, double *out, int slot) {
  __shared__ double red[8];
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < m; i += blockDim.x) acc += partials[i];
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) out[slot] = acc;
}

// fitInterceptCD (fit_linear.nim:28-38) after the dloss sum is in scal[3]
static __global__ void cd_intercept_kernel(double *b, double *yPred, int64_t n, double alpha0, double mu, double *scal,
                                           double *updAbs) {
  const double r = (alpha0 * b[0] + scal[3]) / (mu * (double)n + alpha0);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    yPred[i] -= r;
  if (blockIdx.x == 0 && threadIdx.x == 0) updAbs[0] = fabs(r);
}
static __global__ void cd_intercept_commit_kernel(double *b, double alpha0, double mu, int64_t n, const double *scal) {
  b[0] -= (alpha0 * b[0] + scal[3]) / (mu * (double)n + alpha0);
}

// colNormSq = norm(X, 2, axis=0)^2 (cd.nim:141-142, extmath.nim:151-163): one warp per column
static __global__ void cd_colnorm_kernel(const double *data, const int64_t *indptr, int64_t d, double *out) {
  const int64_t j = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (j >= d) return;
  double acc = 0.0;
  for (int64_t e = indptr[j] + lane; e < indptr[j + 1]; e += 32) acc += data[e] * data[e];
  acc = warp_sum(acc);
  if (lane == 0) {
    const double nr = sqrt(acc);
    out[j] = nr * nr;
  }
}

// ------------------------------------------------------------------ A-cache build (kernels.anova for one component)
// thread per row over the CSR twin; dummy features (d+a, 1.0) follow the row (dataset.nim:182-189)
static __global__ void cd_cache_kernel(const double *data, const int32_t *indices, const int64_t *indptr, int64_t n,
                                       int64_t d, int nAug, const double *Ps, int deg, double *A, int astride) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double a[CD_MAXDEG + 1];
    a[0] = 1.0;
    for (int t = 1; t <= deg; t++) a[t] = 0.0;
    const int64_t rb = indptr[i], re = indptr[i + 1];
    for (int64_t q = rb; q < re + nAug; q++) {
      const double p = q < re ? Ps[indices[q]] : Ps[d + (q - re)];
      const double x = q < re ? data[q] : 1.0;
      if (deg == 2) {
        a[1] += x * p;                     // cacheDeg2[i] += val * P[s, j]   (cd.nim:85-88)
      } else {
        const double t = p * x;
        for (int tt = deg; tt >= 1; tt--) a[tt] += a[tt - 1] * t;   // kernels.nim:31-35
      }
    }
    for (int t = 0; t <= deg; t++) A[i * astride + t] = a[t];
  }
}

// ------------------------------------------------------------------ one batch of coordinate updates
struct CdColArgs {
  const double *data;
  const int32_t *rows;
  const int64_t *indptr;
  const double *y;
  double *yPred, *A, *Ps, *updAbs;   // Ps: the parameter row being swept (P[o][s][:] or w); updAbs indexed by column
  const double *colNormSq;
  int64_t n, d, j0, j1;
  int astride, deg;      // deg: 0 = linear term, 2 = epochDeg2, >2 = epoch
  int loss;
  double thr, mu, reg;   // reg: alpha (linear) or beta (already n-scaled)
  // ---- PCD (optimizer/pcd.nim): per-coordinate prox of the sparsity regulariser
  int prox;              // 0 = none (CD), NIMFM_REG_L1, NIMFM_REG_SQUAREDL12 (chained), NIMFM_REG_SQUAREDL12_ROWS
  int guardAll;          // PCD skips invStepSize < 1e-12 in every sweep (pcd.nim:55,96); CD only for degree <= 2
  int phase;             // 0 = fused; chained prox: 1 = gradient pass only, 2 = refresh pass only
  double gamma;          // n-scaled (pcd.nim:121)
  const double *Po;      // SQUAREDL12_ROWS: the order's P[s'][j] block, to form sum_{s' != s} |P[s'][j]|
  int k, sIdx;
  int64_t dd;
  double *chainA, *chainC, *chainU;   // chained prox, per column: (psj-update)/(1+2lam), 2lam/(1+2lam) (<0: skipped), u
};

__device__ __forceinline__ double cd_soft(double x, double a) {   // softthreshold, regularizer/utils.nim:4-5
  const double m = fabs(x) - a;
  return (x > 0 ? 1.0 : (x < 0 ? -1.0 : 0.0)) * (m > 0.0 ? m : 0.0);
}

template <bool BLOCK_PER_COL>
static __global__ void cd_col_kernel(const CdColArgs a) {
  __shared__ double red[32];
  __shared__ double sh[2];
  const int lane = threadIdx.x & 31;
  int64_t j;
  int tpos, tstep;
  if (BLOCK_PER_COL) {
    j = a.j0 + blockIdx.x;
    tpos = threadIdx.x;
    tstep = blockDim.x;
  } else {
    j = a.j0 + ((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
    tpos = lane;
    tstep = 32;
  }
  if (j >= a.j1) return;
  const bool dummy = j >= a.d;                      // dummy column: every row, value 1.0 (dataset.nim:245-252)
  const int64_t cb = dummy ? 0 : a.indptr[j];
  const int64_t len = dummy ? a.n : a.indptr[j + 1] - cb;
  const double psj = a.Ps[j];
  const int deg = a.deg;
  const bool leader = BLOCK_PER_COL ? threadIdx.x == 0 : lane == 0;
  double u, pnew = 0.0;
  if (a.phase != 2) {
    // ---- pass 1: gradient and curvature (update(), cd.nim:36-47 / cd.nim:93-97 / fit_linear.nim:14-17)
    double upd = 0.0, inv = 0.0;
    for (int64_t e = tpos; e < len; e += tstep) {
      const int64_t i = dummy ? e : (int64_t)a.rows[cb + e];
      const double x = dummy ? 1.0 : a.data[cb + e];
      double g;
      if (deg == 0) {
        g = x;
      } else if (deg == 2) {
        g = (a.A[i * a.astride + 1] - psj * x) * x;
      } else {
        g = x;                                         // computeDerivative, cd.nim:29-33
        for (int t = 1; t < deg; t++) g = x * (a.A[i * a.astride + t] - psj * g);
      }
      upd += dev_dloss(a.loss, a.thr, a.y[i], a.yPred[i]) * g;
      inv += g * g;
    }
    if (BLOCK_PER_COL) {
      upd = block_sum(upd, red);
      __syncthreads();
      inv = block_sum(inv, red);
      if (threadIdx.x == 0) {
        sh[0] = upd;
        sh[1] = inv;
      }
      __syncthreads();
      upd = sh[0];
      inv = sh[1];
    } else {
      upd = warp_sum(upd);
      inv = warp_sum(inv);
    }
    upd += a.reg * psj;
    if (deg == 0) inv = a.mu * a.colNormSq[j] + a.reg;   // fit_linear.nim:18
    else inv = inv * a.mu + a.reg;
    // the guard exists in epochDeg2 / fitLinearCD, and in both sweeps of PCD (pcd.nim:55,96)
    const bool skip = (deg <= 2 || a.guardAll) && inv < 1e-12;
    if (a.phase == 1) {                                  // chained prox: hand (a_j, c_j) to pcd_chain_kernel
      if (leader) {
        const double lam = a.gamma / inv, den = 1 + 2 * lam;
        a.chainA[j] = skip ? 0.0 : (psj - upd / inv) / den;
        a.chainC[j] = skip ? -1.0 : 2 * lam / den;
      }
      return;
    }
    if (skip) {
      if (leader) a.updAbs[j] = 0.0;
      return;
    }
    u = upd / inv;
    if (deg != 0 && a.prox == NIMFM_REG_L1) {            // l1.nim:22-24
      pnew = cd_soft(psj - u, a.gamma / inv);
      u = psj - pnew;
    } else if (deg != 0 && a.prox == NIMFM_REG_SQUAREDL12_ROWS) {   // squaredl12.nim:108-114, transpose=false
      double dcache = 0.0;
      for (int s2 = 0; s2 < a.k; s2++)
        if (s2 != a.sIdx) dcache += fabs(a.Po[(int64_t)s2 * a.dd + j]);
      const double lam = a.gamma / inv;
      pnew = cd_soft((psj - u) / (1 + 2 * lam), 2 * lam * dcache / (1 + 2 * lam));
      u = psj - pnew;
    } else {
      pnew = psj - u;
    }
  } else {
    if (a.chainC[j] < 0.0) return;                       // skipped coordinate: P stays, the chain zeroed updAbs
    u = a.chainU[j];
  }
  // ---- pass 2: in-place refresh over the column (cd.nim:67-73 / :104-106 / fit_linear.nim:24-25)
  for (int64_t e = tpos; e < len; e += tstep) {
    const int64_t i = dummy ? e : (int64_t)a.rows[cb + e];
    const double x = dummy ? 1.0 : a.data[cb + e];
    if (deg == 0) {
      a.yPred[i] -= u * x;
    } else if (deg == 2) {
      double *c = a.A + i * a.astride + 1;
      a.yPred[i] -= u * (*c - psj * x) * x;
      *c -= u * x;
    } else {
      double *Ai = a.A + i * a.astride;
      double prev = x;                                 // dA[0]
      for (int t = 1; t < deg; t++) {
        const double cur = x * (Ai[t] - psj * prev);   // dA[t] from the OLD A[i,t]
        Ai[t] -= u * prev;
        prev = cur;
      }
      Ai[deg] -= u * prev;
      a.yPred[i] -= u * prev;
    }
  }
  if (leader) {
    if (a.phase == 0) {
      a.Ps[j] = pnew;                                  // CD: psj - u; PCD: exactly the prox result
      a.updAbs[j] = fabs(u);
    } else {
      a.Ps[j] = a.chainA[j];                           // the chain's prox result
    }
  }
}

// The chained prox of SquaredL12(transpose=true) (squaredl12.nim:108-114,182-185): coordinate j's
// threshold depends on cache = sum_j' |P[s][j']| as left by every earlier coordinate of the sweep, so
// the batch's columns are resolved in order by ONE warp (all lanes carry the same running cache; lane t
// keeps column base+t's result).  In: a_j, c_j from phase 1.  Out: the new P[s][j] (in chainA), u_j, |u_j|.
static __global__ void pcd_chain_kernel(const double *Ps, double *chainA, const double *chainC, double *chainU,
                                        double *updAbs, int64_t j0, int64_t j1, double *cache) {
  const int lane = threadIdx.x & 31;
  double c = *cache;
  for (int64_t base = j0; base < j1; base += 32) {
    const int64_t j = base + lane;
    const double aj = j < j1 ? chainA[j] : 0.0, cj = j < j1 ? chainC[j] : -1.0, pj = j < j1 ? Ps[j] : 0.0;
    double myU = 0.0, myP = pj;
    const int cnt = (int)min((int64_t)32, j1 - base);
    for (int t = 0; t < cnt; ++t) {
      const double at = __shfl_sync(0xffffffffu, aj, t), ct = __shfl_sync(0xffffffffu, cj, t),
                   pt = __shfl_sync(0xffffffffu, pj, t);
      if (ct >= 0.0) {
        const double ap = fabs(pt);
        const double pn = cd_soft(at, ct * (c - ap));    // dcache = cache - absp[j]
        c -= ap;                                         // updateCacheCD
        c += fabs(pn);
        if (lane == t) { myU = pt - pn; myP = pn; }
      }
    }
    if (j < j1 && cj >= 0.0) {
      chainA[j] = myP;        // committed to P by the refresh pass, which still needs the old value
      chainU[j] = myU;
      updAbs[j] = fabs(myU);
    } else if (j < j1) {
      updAbs[j] = 0.0;
    }
  }
  if (lane == 0) *cache = c;
}

static __global__ void pcd_abs_sum_kernel(const double *v, int64_t n, double *out) {   // computeCacheCD: sum(absp)
  __shared__ double red[8];
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc += fabs(v[i]);
  acc = block_sum(acc, red);
  if (threadIdx.x == 0) *out = acc;
}

static int cd_reduce(nimfm_ctx *ctx, int kind, const double *v0, const double *v1, int64_t n, int loss, double thr,
                     double *scal, int slot) {
  const int grid = (int)std::min<int64_t>(1024, std::max<int64_t>(1, (n + 255) / 256));
  int rc = nimfm_ensure_partials(ctx, 1024);
  if (rc) return rc;
  if (kind == 0) cd_sum_dloss_kernel<<<grid, 256, 0, ctx->stream>>>(v0, v1, n, loss, thr, ctx->partials);
  else if (kind == 1) cd_sum_loss_kernel<<<grid, 256, 0, ctx->stream>>>(v0, v1, n, loss, thr, ctx->partials);
  else cd_sumsq_kernel<<<grid, 256, 0, ctx->stream>>>(v0, n, ctx->partials);
  cd_final_sum_kernel<<<1, 256, 0, ctx->stream>>>(ctx->partials, grid, scal, slot);
  ctx->launches += 2;
  return NIMFM_OK;
}

struct PcdProx {   // sparsity regulariser of a PCD sweep (zeros == plain CD)
  int prox = 0, guardAll = 0;
  double gamma = 0.0;
  const double *Po = nullptr;
  int k = 0, sIdx = 0;
};

// blockThreads: threads of a block-per-column launch (long columns), 0 = one warp per column
static void cd_launch_cols(nimfm_ctx *ctx, const CdColArgs &a, int blockThreads) {
  const int64_t cols = a.j1 - a.j0;
  if (blockThreads > 0) {
    cd_col_kernel<true><<<(int)cols, blockThreads, 0, ctx->stream>>>(a);
  } else {
    const int64_t threads = cols * 32;
    cd_col_kernel<false><<<(int)((threads + 127) / 128), 128, 0, ctx->stream>>>(a);
  }
  LAUNCHED(ctx);
}

static int cd_sweep(nimfm_ctx *ctx, CdState *st, const nimfm_dataset *X, nimfm_fm *fm, const nimfm_cd_cfg *cfg,
                    double *Ps, int deg, double reg, double *updAbs, int64_t nCols, const PcdProx &px, double *Abuf) {
  // nCols == d for the linear sweep (dummy features removed, cd.nim:159), d + nAug otherwise
  CdColArgs a;
  memset(&a, 0, sizeof(a));
  a.data = X->data; a.rows = X->indices; a.indptr = X->indptr; a.y = X->y;
  a.yPred = fm->yPred; a.A = Abuf; a.Ps = Ps; a.updAbs = updAbs; a.colNormSq = fm->colNormSq;
  a.n = X->n; a.d = X->d; a.astride = fm->degree + 1; a.deg = deg;
  a.loss = cfg->loss; a.thr = cfg->huberThreshold; a.mu = loss_mu(cfg->loss); a.reg = reg;
  a.prox = deg == 0 ? 0 : px.prox; a.guardAll = px.guardAll; a.gamma = px.gamma;
  a.Po = px.Po; a.k = px.k; a.sIdx = px.sIdx; a.dd = fm->dd();
  const bool chained = a.prox == NIMFM_REG_SQUAREDL12;
  double *cache = fm->cdScal + 8;
  if (chained) {
    a.chainA = st->chain; a.chainC = st->chain + a.dd; a.chainU = st->chain + 2 * a.dd;
    pcd_abs_sum_kernel<<<1, 256, 0, ctx->stream>>>(Ps, nCols, cache);   // computeCacheCD (squaredl12.nim:173-179)
    LAUNCHED(ctx);
  }
  auto run = [&](int blockPerCol) {
    if (!chained) {
      a.phase = 0;
      cd_launch_cols(ctx, a, blockPerCol);
      return;
    }
    a.phase = 1;
    cd_launch_cols(ctx, a, blockPerCol);
    pcd_chain_kernel<<<1, 32, 0, ctx->stream>>>(Ps, a.chainA, a.chainC, a.chainU, updAbs, a.j0, a.j1, cache);
    LAUNCHED(ctx);
    a.phase = 2;
    cd_launch_cols(ctx, a, blockPerCol);
  };
  const size_t nb = st->batchStart.size() - 1;
  for (size_t b = 0; b < nb; b++) {
    a.j0 = st->batchStart[b];
    a.j1 = st->batchStart[b + 1];
    // column length decides the shape: a warp walks a 100-row column in 4 dependent round trips per pass,
    // a 128-thread block in one (the sweep is latency-bound: ~100 short kernels per outer iteration)
    const int64_t mx = st->batchMaxLen[b];
    run(mx > 2048 ? 1024 : (mx > 256 ? 256 : (mx > 48 ? 128 : 0)));
  }
  for (int64_t j = X->d; j < nCols; j++) {   // dummy columns touch every row: one batch each
    a.j0 = j;
    a.j1 = j + 1;
    run(1024);
  }
  return NIMFM_OK;
}

static int cd_epoch_impl(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_cd_cfg *cfg, int prox,
                         double gammaRaw, double *viol, double *lossMean, double *regOverN);
static int cd_enqueue_epoch(nimfm_ctx *ctx, CdState *st, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_cd_cfg *cfg,
                            int prox, double gammaRaw);

extern "C" {

int32_t nimfm_fm_cd_begin(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_cd_cfg *cfg) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(fm && X && cfg, "NULL argument");
  REQUIRE(X->kind == NIMFM_DS_CSC, "CD needs a CSCDataset (ColDataset)");
  REQUIRE(X->d == fm->d, "Invalid nFeatures.");
  REQUIRE(X->y != nullptr, "dataset has no targets (nimfm_dataset_set_targets)");
  CK(cudaSetDevice(ctx->device));
  const int64_t n = X->n, d = X->d, dd = fm->dd(), nP = fm->nP();
  CdState *st = cd_state(fm, true);
  st->alpha0 = cfg->alpha0 * (double)n;   // cd.nim:123-125
  st->alpha = cfg->alpha * (double)n;
  st->beta = cfg->beta * (double)n;
  int rc;
  if (st->csr) nimfm_dataset_free(ctx, st->csr);
  st->csr = nullptr;
  if (st->graph) cudaGraphExecDestroy(st->graph);   // a new fit: buffers are reallocated below
  st->graph = nullptr;
  if ((rc = nimfm_dataset_transpose(ctx, X, &st->csr))) return rc;
  // ---- batches of consecutive, pairwise row-disjoint columns
  {
    std::vector<int32_t> rows((size_t)X->nnz);
    std::vector<int64_t> ptr((size_t)d + 1);
    CK(cudaMemcpy(rows.data(), X->indices, (size_t)X->nnz * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(ptr.data(), X->indptr, ((size_t)d + 1) * 8, cudaMemcpyDeviceToHost));
    std::vector<int64_t> mark((size_t)std::max<int64_t>(n, 1), -1);
    st->batchStart.clear();
    st->batchMaxLen.clear();
    int64_t cur = -1;
    for (int64_t j = 0; j < d; j++) {
      bool conflict = cur < 0;
      for (int64_t e = ptr[j]; e < ptr[j + 1] && !conflict; e++)
        if (mark[rows[e]] == cur) conflict = true;
      if (conflict) {
        cur = (int64_t)st->batchStart.size();
        st->batchStart.push_back(j);
        st->batchMaxLen.push_back(0);
      }
      for (int64_t e = ptr[j]; e < ptr[j + 1]; e++) mark[rows[e]] = cur;
      st->batchMaxLen.back() = std::max(st->batchMaxLen.back(), ptr[j + 1] - ptr[j]);
    }
    st->batchStart.push_back(d);
  }
  // ---- caches
  for (double *p : {fm->Pcm, fm->yPred, fm->Acache, fm->colNormSq, fm->cdScal}) cudaFree(p);
  fm->Pcm = fm->yPred = fm->Acache = fm->colNormSq = fm->cdScal = nullptr;
  CK(cudaMalloc(&fm->Pcm, (size_t)std::max<int64_t>(nP, 1) * 8));
  CK(cudaMalloc(&fm->yPred, (size_t)std::max<int64_t>(n, 1) * 8));
  CK(cudaMalloc(&fm->Acache, (size_t)std::max<int64_t>(n, 1) * (fm->degree + 1) * 8 * 2));   // double buffer
  CK(cudaMalloc(&fm->colNormSq, (size_t)d * 8));
  CK(cudaMalloc(&fm->cdScal, 16 * 8));
  CK(cudaMemsetAsync(fm->cdScal, 0, 16 * 8, ctx->stream));
  const int64_t nUpd = 1 + d + (int64_t)fm->nOrders * fm->k * dd;
  if (st->updCap < nUpd) {
    cudaFree(st->updAbs);
    CK(cudaMalloc(&st->updAbs, (size_t)nUpd * 8));
    st->updCap = nUpd;
  }
  fm->cdN = n;
  if (nP > 0) {   // degree 1: no P
    cd_permute_kernel<<<ew_grid(ctx, nP), 256, 0, ctx->stream>>>(fm->P, fm->Pcm, fm->nOrders, fm->k, dd, 1);
    LAUNCHED(ctx);
  }
  if (fm->fitLinear) {
    cd_colnorm_kernel<<<(int)((d * 32 + 127) / 128), 128, 0, ctx->stream>>>(X->data, X->indptr, d, fm->colNormSq);
    LAUNCHED(ctx);
  }
  // yPred = linear + intercept + sum anova (cd.nim:144-151)
  if ((rc = nimfm_fm_predict_device(ctx, fm, st->csr, fm->yPred))) return rc;
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  fm->cdReady = true;
  return NIMFM_OK;
}

int32_t nimfm_fm_cd_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_cd_cfg *cfg, double *viol,
                          double *lossMean, double *regOverN) {
  return cd_epoch_impl(ctx, fm, X, cfg, 0, 0.0, viol, lossMean, regOverN);
}

// One outer iteration of PCD.fit (pcd.nim:156-172): cd.fit's sweeps with the per-coordinate prox of the
// sparsity regulariser and the invStepSize guard in every sweep.  regOverN excludes gamma*reg.eval
// (the host adds it when it prints, :181-183).
int32_t nimfm_fm_pcd_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_pcd_cfg *cfg, double *viol,
                           double *lossMean, double *regOverN) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(cfg != nullptr, "NULL argument");
  REQUIRE(cfg->reg == NIMFM_REG_L1 || cfg->reg == NIMFM_REG_SQUAREDL12 || cfg->reg == NIMFM_REG_SQUAREDL12_ROWS,
          "PCD supports the L1 and SquaredL12 regularisers");
  // SquaredL12.initCD raises for degree != 2 (squaredl12.nim:90-93)
  REQUIRE(!(cfg->reg != NIMFM_REG_L1 && fm && fm->degree != 2), "SquaredL12 supports only degree=2.");
  nimfm_cd_cfg c;
  c.loss = cfg->loss; c.huberThreshold = cfg->huberThreshold;
  c.alpha0 = cfg->alpha0; c.alpha = cfg->alpha; c.beta = cfg->beta;
  return cd_epoch_impl(ctx, fm, X, &c, cfg->reg, cfg->gamma, viol, lossMean, regOverN);
}

}  // extern "C"

static int cd_epoch_impl(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_cd_cfg *cfg, int prox,
                         double gammaRaw, double *viol, double *lossMean, double *regOverN) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(fm && X && cfg, "NULL argument");
  if (!fm->cdReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_fm_cd_begin was not called");
  CdState *st = cd_state(fm, false);
  REQUIRE(st && X->kind == NIMFM_DS_CSC && X->n == fm->cdN && X->d == fm->d, "dataset does not match cd_begin");
  CK(cudaSetDevice(ctx->device));
  const int64_t n = X->n, dd = fm->dd();
  int rc;
  if ((rc = nimfm_ensure_partials(ctx, 1024))) return rc;            // no allocation inside a capture
  if (prox == NIMFM_REG_SQUAREDL12 && st->chainCap < 3 * dd) {
    cudaFree(st->chain);
    st->chain = nullptr;
    CK(cudaMalloc(&st->chain, (size_t)(3 * dd) * 8));
    st->chainCap = 3 * dd;
  }
  const char *genv = getenv("NIMFM_CD_GRAPH");
  const bool useGraph = !(genv && genv[0] == '0');
  const CdState::Key key = {prox, cfg->loss, gammaRaw, cfg->huberThreshold, st->alpha0, st->alpha, st->beta};
  if (!useGraph) {
    if ((rc = cd_enqueue_epoch(ctx, st, fm, X, cfg, prox, gammaRaw))) return rc;
  } else {
    if (st->graph && memcmp(&key, &st->graphKey, sizeof(key)) != 0) {
      cudaGraphExecDestroy(st->graph);
      st->graph = nullptr;
    }
    if (!st->graph) {
      const int64_t l0 = ctx->launches;
      CK(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
      rc = cd_enqueue_epoch(ctx, st, fm, X, cfg, prox, gammaRaw);
      cudaGraph_t g = nullptr;
      cudaError_t ce = cudaStreamEndCapture(ctx->stream, &g);
      st->graphKernels = ctx->launches - l0;
      ctx->launches = l0;
      if (rc) { if (g) cudaGraphDestroy(g); return rc; }
      if (ce != cudaSuccess) return nimfm_fail(ctx, NIMFM_ERR_CUDA, "CD graph capture: %s", cudaGetErrorString(ce));
      ce = cudaGraphInstantiate(&st->graph, g, 0);
      cudaGraphDestroy(g);
      if (ce != cudaSuccess) return nimfm_fail(ctx, NIMFM_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ce));
      st->graphKey = key;
    }
    CK(cudaGraphLaunch(st->graph, ctx->stream));
    ctx->launches += st->graphKernels;
  }
  CK(cudaGetLastError());
  double h[8];
  CK(cudaMemcpyAsync(ctx->hostScalars, fm->cdScal, 64, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(ctx->hostScalars + 8, fm->b, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  memcpy(h, ctx->hostScalars, 64);
  const double hb = ctx->hostScalars[8];
  if (viol) *viol = h[0];
  if (lossMean) *lossMean = h[1] / (double)n;
  if (regOverN) {
    // regularization (optimizer/utils.nim:56-59): norm(.,2)^2 == sqrt(sum sq)^2
    const double nw = sqrt(h[4]), np = sqrt(h[5]);
    const double reg = 0.5 * st->alpha0 * (hb * hb) + 0.5 * st->alpha * (nw * nw) + 0.5 * st->beta * (np * np);
    *regOverN = reg / (double)n;
  }
  return NIMFM_OK;
}

// every kernel of one outer iteration, enqueued on ctx->stream (no synchronisation, no allocation)
static int cd_enqueue_epoch(nimfm_ctx *ctx, CdState *st, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_cd_cfg *cfg,
                            int prox, double gammaRaw) {
  const int64_t n = X->n, d = X->d, dd = fm->dd();
  const double mu = loss_mu(cfg->loss);
  const int64_t nUpd = 1 + d + (int64_t)fm->nOrders * fm->k * dd;
  int rc;
  CK(cudaMemsetAsync(st->updAbs, 0, (size_t)nUpd * 8, ctx->stream));
  const int rowGrid = ew_grid(ctx, n);
  if (fm->fitIntercept) {                                            // fitInterceptCD
    if ((rc = cd_reduce(ctx, 0, X->y, fm->yPred, n, cfg->loss, cfg->huberThreshold, fm->cdScal, 3))) return rc;
    cd_intercept_kernel<<<rowGrid, 256, 0, ctx->stream>>>(fm->b, fm->yPred, n, st->alpha0, mu, fm->cdScal, st->updAbs);
    cd_intercept_commit_kernel<<<1, 1, 0, ctx->stream>>>(fm->b, st->alpha0, mu, n, fm->cdScal);
    ctx->launches += 2;
  }
  PcdProx px;
  px.prox = prox;
  px.guardAll = prox != 0;
  px.gamma = gammaRaw * (double)n;                                   // pcd.nim:121
  px.k = fm->k;
  if (fm->fitLinear)                                                 // fitLinearCD (dummy features removed)
    if ((rc = cd_sweep(ctx, st, X, fm, cfg, fm->w, 0, st->alpha, st->updAbs + 1, d, px, fm->Acache))) return rc;
  const nimfm_dataset *R = st->csr;
  // The A-cache of sweep t+1 depends only on P[t+1] and X, not on what sweep t writes, so it is built
  // on a second stream into the other half of a double buffer WHILE sweep t runs (a fork/join inside the
  // captured graph): one kernel of every three leaves the critical path.
  const int T = fm->nOrders * fm->k;
  const int astride = fm->degree + 1;
  const size_t aHalf = (size_t)std::max<int64_t>(n, 1) * astride;
  cudaStream_t side = ctx->copyStream;
  auto build_cache = [&](int t, cudaStream_t strm) {
    const int o = t / fm->k;
    double *Ps = fm->Pcm + (int64_t)t * dd;
    cd_cache_kernel<<<rowGrid, 256, 0, strm>>>(R->data, R->indices, R->indptr, n, d, fm->nAug, Ps, fm->degree - o,
                                               fm->Acache + (size_t)(t & 1) * aHalf, astride);
    LAUNCHED(ctx);
  };
  if (T > 0) build_cache(0, ctx->stream);
  for (int t = 0; t < T; t++) {
    const int o = t / fm->k, sIdx = t - o * fm->k;
    if (t + 1 < T) {
      CK(cudaEventRecord(ctx->evCopied[0], ctx->stream));      // sweep t-1 (last user of the other half) is done
      CK(cudaStreamWaitEvent(side, ctx->evCopied[0], 0));
      build_cache(t + 1, side);
      CK(cudaEventRecord(ctx->evCopied[1], side));
    }
    px.Po = fm->Pcm + (int64_t)o * fm->k * dd;
    px.sIdx = sIdx;
    double *Ps = fm->Pcm + (int64_t)t * dd;
    double *upd = st->updAbs + 1 + d + (int64_t)t * dd;
    if ((rc = cd_sweep(ctx, st, X, fm, cfg, Ps, fm->degree - o, st->beta, upd, dd, px,
                       fm->Acache + (size_t)(t & 1) * aHalf)))
      return rc;
    if (t + 1 < T) CK(cudaStreamWaitEvent(ctx->stream, ctx->evCopied[1], 0));
  }
  // viol (fixed-order sum of |update|), mean loss, regularization / n (cd.nim:177-184)
  int grid = (int)std::min<int64_t>(1024, std::max<int64_t>(1, (nUpd + 255) / 256));
  if ((rc = nimfm_ensure_partials(ctx, 1024))) return rc;
  cd_final_sum_kernel<<<1, 256, 0, ctx->stream>>>(st->updAbs, nUpd, fm->cdScal, 0);
  LAUNCHED(ctx);
  (void)grid;
  if ((rc = cd_reduce(ctx, 1, X->y, fm->yPred, n, cfg->loss, cfg->huberThreshold, fm->cdScal, 1))) return rc;
  if ((rc = cd_reduce(ctx, 2, fm->w, nullptr, d, 0, 0, fm->cdScal, 4))) return rc;
  if (fm->nP() == 0) {   // degree 1: no P, ||P||^2 = 0
    CK(cudaMemsetAsync(fm->cdScal + 5, 0, 8, ctx->stream));
    return NIMFM_OK;
  }
  if ((rc = cd_reduce(ctx, 2, fm->Pcm, nullptr, fm->nP(), 0, 0, fm->cdScal, 5))) return rc;
  // keep the feature-major copy current so get_params / callbacks see this epoch's parameters
  cd_permute_kernel<<<ew_grid(ctx, fm->nP()), 256, 0, ctx->stream>>>(fm->P, fm->Pcm, fm->nOrders, fm->k, dd, 0);
  LAUNCHED(ctx);
  return NIMFM_OK;
}

extern "C" {

int32_t nimfm_fm_cd_get_ypred(nimfm_ctx *ctx, nimfm_fm *fm, double *yPred) {
  if (!ctx || !fm || !yPred) return NIMFM_ERR_INVALID;
  if (!fm->cdReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_fm_cd_begin was not called");
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpy(yPred, fm->yPred, (size_t)fm->cdN * 8, cudaMemcpyDeviceToHost));
  return NIMFM_OK;
}

int32_t nimfm_fm_cd_end(nimfm_ctx *ctx, nimfm_fm *fm) {
  if (!ctx || !fm) return NIMFM_ERR_INVALID;
  if (!fm->cdReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_fm_cd_begin was not called");
  CK(cudaSetDevice(ctx->device));
  if (fm->nP() > 0) {
    cd_permute_kernel<<<ew_grid(ctx, fm->nP()), 256, 0, ctx->stream>>>(fm->P, fm->Pcm, fm->nOrders, fm->k, fm->dd(), 0);
    LAUNCHED(ctx);
  }
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  CdState *st = cd_state(fm, false);
  if (st) {
    nimfm_dataset_free(ctx, st->csr);
    cudaFree(st->updAbs);
    cudaFree(st->chain);
    if (st->graph) cudaGraphExecDestroy(st->graph);
    for (size_t i = 0; i < g_cd.size(); i++)
      if (g_cd[i].first == fm) {
        delete g_cd[i].second;
        g_cd.erase(g_cd.begin() + i);
        break;
      }
  }
  fm->cdReady = false;
  return NIMFM_OK;
}

}  // extern "C"
