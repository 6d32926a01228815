// fm_linear.cu -- the row kernel of the degree-1 FM: the linear model yhat = b + <w, x> (nOrders = 0, no P, no
// dummy features; factorization_machine.nim:89-97).  plan_rows (fm_api.cu) selects it for every row-parallel entry
// point when the model has no ANOVA term, so decisionFunction (resident, host-fed, stream windows), predict+grad,
// the MBPSGD / minibatch-SGD gradients, minibatch AdaGrad and the deterministic route's forward all run it with the
// RowArgs / partials contract of fm_rows.cuh unchanged.
//
// A degree-1 row is an SpMV row: a group of L lanes (L in {4, 8, 16, 32}, the smallest width that covers the
// dataset's longest row, capped at one warp) owns one row, the lanes stride over its nonzeros, gather w[j] * x and
// reduce with shuffles; the group's first lane adds the intercept and evaluates the loss.  No shared-memory staging:
// each nonzero is read once for the forward and once more (from L1) for the backward.  (w is read-only in every
// mode: the gradients go to separate buffers.)
//   MODE_PREDICT  yOut[q] = yhat
//   MODE_GRAD     gw[j] += coef * x with FP64 REDs, coef = dloss / mb (minibatch_psgd.nim:73-85)
//   MODE_ADAGRAD  g = dloss * x rounded on its own; gw[j] += g, dGnw[j] += g * g (adagrad.nim:113-124); the
//                 intercept of the batch comes from g_sum / g_norm as in fm_rows_kernel's AdaGrad prologue
//   MODE_STASH    the row's coef goes to its stash record (fm_cols.cu: the deterministic route's column pass
//                 fm_cols_linear_kernel adds coef * x per column in ascending row order)
// Hot features (dataset.cu: columns in >= 1/16 of a row sample, at most 16): their w-gradients are summed per lane
// in shared memory ([slot][lane], one column per lane: no shared atomics) and flushed with one RED per slot and
// warp when the kernel ends, as fm_rows_kernel does, instead of ~nRows REDs on one address.
// Every mode writes the per-warp partials (loss, sum coef, sum dL^2, 0) that reduce_partials_kernel reads.
#include "fm_rows.cuh"

namespace {

template <int MODE, int L>
__global__ void __launch_bounds__(256, 4) fm_linear_rows_kernel(const RowArgs a) {
  constexpr bool BACK = MODE == MODE_GRAD || MODE == MODE_ADAGRAD;
  constexpr int NACC = MODE == MODE_ADAGRAD ? 2 : 1;
  constexpr int GPW = 32 / L;   // rows per warp
  extern __shared__ __align__(16) unsigned char lin_smem[];
  const int lane = threadIdx.x & 31, warpInBlock = threadIdx.x >> 5;
  const int gl = lane & (L - 1), gid = lane / L;
  const int nHot = BACK ? a.nHot : 0;
  double *hot = reinterpret_cast<double *>(lin_smem) + (size_t)warpInBlock * nHot * 32 * NACC;   // [NACC][nHot][32]
  for (int s = 0; s < nHot * NACC; ++s) hot[s * 32 + lane] = 0.0;

  const int warpsPerBlock = blockDim.x >> 5;
  const int64_t warpGlobal = (int64_t)blockIdx.x * warpsPerBlock + warpInBlock;
  const int64_t nWarps = (int64_t)gridDim.x * warpsPerBlock;
  const int64_t tiles = (a.nRows + GPW - 1) / GPW;

  double bias = a.b[0];
  if (MODE == MODE_ADAGRAD && !a.first && a.fitIntercept) {   // adagrad.nim:101-105
    const double den = sqrt(a.adaScal[1]) + a.eta0 * a.tIt * a.alpha0;
    bias = -a.eta0 * a.adaScal[0] / den;
  }
  double accLoss = 0.0, accB1 = 0.0, accB2 = 0.0;

  for (int64_t tile = warpGlobal; tile < tiles; tile += nWarps) {
    const int64_t q = tile * GPW + gid;
    const bool active = q < a.nRows;
    int64_t r = 0, rb = 0;
    int z = 0;
    if (active) {
      r = a.rowIdx ? (int64_t)a.rowIdx[q] : (a.rowBegin + q) % a.n;
      rb = a.indptr[r];
      z = (int)(a.indptr[r + 1] - rb);
    }
    // two nonzeros per lane and step: both index loads, then both gathers, in flight together (same order of adds)
    double lin = 0.0;
    for (int u = gl; u < z; u += 2 * L) {
      const bool two = u + L < z;
      const int j0 = __ldg(a.indices + rb + u), j1 = two ? __ldg(a.indices + rb + u + L) : 0;
      const double x0 = __ldg(a.data + rb + u), x1 = two ? __ldg(a.data + rb + u + L) : 0.0;
      lin += __ldg(a.w + j0) * x0;
      if (two) lin += __ldg(a.w + j1) * x1;
    }
    const double yhat = bias + group_sum(lin, L);
    if (!active) continue;   // (no shuffles below)
    if (a.yOut && gl == 0) a.yOut[q] = yhat;
    if (MODE == MODE_PREDICT) continue;
    const double yi = a.y[r];
    const double dL = dev_dloss(a.loss, a.thr, yi, yhat);
    const double coef = MODE == MODE_ADAGRAD ? dL : dL / a.mb;
    if (gl == 0) {
      accLoss += dev_loss(a.loss, a.thr, yi, yhat);
      accB1 += coef;
      accB2 += dL * dL;
      if (MODE == MODE_STASH) a.stash[(size_t)q * a.stashStride] = coef;
    }
    if (BACK && a.fitLinear) {
      for (int u = gl; u < z; u += L) {
        const int j = a.indices[rb + u];
        const double gx = __dmul_rn(coef, a.data[rb + u]);
        const int slot = nHot > 0 ? (int)a.hotSlot[j] : NIMFM_COLD;
        if (slot != NIMFM_COLD) {
          hot[slot * 32 + lane] += gx;
          if (MODE == MODE_ADAGRAD) hot[(nHot + slot) * 32 + lane] += __dmul_rn(gx, gx);
        } else {
          atomicAdd(a.gw + j, gx);
          if (MODE == MODE_ADAGRAD) atomicAdd(a.dGnw + j, __dmul_rn(gx, gx));
        }
      }
    }
  }

  if (BACK && nHot > 0) {   // uniform across the warp: every lane takes part in the sums
    for (int s = 0; s < nHot; ++s) {
      const double v = warp_sum(hot[s * 32 + lane]);
      const double v2 = MODE == MODE_ADAGRAD ? warp_sum(hot[(nHot + s) * 32 + lane]) : 0.0;
      if (lane == 0 && a.fitLinear) {
        const int64_t j = a.hotList[s];
        if (v != 0.0) atomicAdd(a.gw + j, v);
        if (MODE == MODE_ADAGRAD && v2 != 0.0) atomicAdd(a.dGnw + j, v2);
      }
    }
  }
  if (MODE != MODE_PREDICT) {
    accLoss = warp_sum(accLoss);
    accB1 = warp_sum(accB1);
    accB2 = warp_sum(accB2);
    if (lane == 0) {
      a.partials[warpGlobal * 4 + 0] = accLoss;
      a.partials[warpGlobal * 4 + 1] = accB1;
      a.partials[warpGlobal * 4 + 2] = accB2;
      a.partials[warpGlobal * 4 + 3] = 0.0;
    }
  }
}

template <int MODE>
RowKernel linear_kernel_of(int L) {
  switch (L) {
    case 4: return fm_linear_rows_kernel<MODE, 4>;
    case 8: return fm_linear_rows_kernel<MODE, 8>;
    case 16: return fm_linear_rows_kernel<MODE, 16>;
    default: return fm_linear_rows_kernel<MODE, 32>;
  }
}

}  // namespace

// The launch of the linear row kernel for nRows rows of X: group width from the longest row, 256-thread blocks,
// a persistent grid of occupancy x numSMs blocks at most.  pl->stream = false (the lazy MBPSGD / minibatch-SGD
// epochs, which fold shrink factors into the streaming kernel's x, decline), pl->G = lanes per row, pl->CH = 0.
int nimfm_fm_linear_plan(nimfm_ctx *ctx, const nimfm_dataset *X, int64_t nRows, int mode, RowPlan *pl) {
  int L = 4;
  while (L < 32 && L < X->maxSegNnz) L <<= 1;
  RowKernel kern;
  switch (mode) {
    case MODE_PREDICT: kern = linear_kernel_of<MODE_PREDICT>(L); break;
    case MODE_GRAD: kern = linear_kernel_of<MODE_GRAD>(L); break;
    case MODE_ADAGRAD: kern = linear_kernel_of<MODE_ADAGRAD>(L); break;
    default: kern = linear_kernel_of<MODE_STASH>(L); break;
  }
  const int nAcc = mode == MODE_ADAGRAD ? 2 : (mode == MODE_GRAD ? 1 : 0);
  const int nHot = X->hotSlot ? X->nHot : 0;
  const int block = 256;
  const size_t smem = (size_t)(block / 32) * nHot * 32 * nAcc * 8;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, block, smem));
  if (occ < 1) return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "linear row kernel does not fit on an SM");
  const int64_t tiles = (nRows + (32 / L) - 1) / (32 / L);
  int64_t grid = (tiles + block / 32 - 1) / (block / 32);
  const int64_t cap = (int64_t)occ * ctx->numSMs;
  if (grid > cap) grid = cap;
  if (grid < 1) grid = 1;
  pl->kern = kern;
  pl->stream = false;
  pl->G = L;
  pl->CH = 0;
  pl->block = block;
  pl->smem = smem;
  pl->grid = (int)grid;
  pl->nWarps = grid * (block / 32);
  return NIMFM_OK;
}
