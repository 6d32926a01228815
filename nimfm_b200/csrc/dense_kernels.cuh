// dense_kernels.cuh -- small dense / reduction kernels shared by the FM and FFM entry points:
// fixed-order partial reduction, the MBPSGD dense step (K3) and the AdaGrad dense passes (K5).
#pragma once
#include "common.cuh"

static inline int ew_grid(nimfm_ctx *ctx, int64_t n, int block = 256) {
  int64_t g = (n + block - 1) / block;
  int64_t cap = (int64_t)ctx->numSMs * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

// ------------------------------------------------------------------ small reductions
// sums partials[nRows4][4] column-wise in a fixed order; out[c] (+)= sum
static __global__ void reduce_partials_kernel(const double *partials, int64_t rows, double *out, int accumulate) {
  __shared__ double red[8];
  double acc[4] = {0, 0, 0, 0};
  for (int64_t r = threadIdx.x; r < rows; r += blockDim.x) {
#pragma unroll
    for (int c = 0; c < 4; c++) acc[c] += partials[r * 4 + c];
  }
#pragma unroll
  for (int c = 0; c < 4; c++) {
    double v = block_sum(acc[c], red);
    if (threadIdx.x == 0) out[c] = accumulate ? out[c] + v : v;
    __syncthreads();
  }
}

// ------------------------------------------------------------------ MBPSGD dense step (K3)
// Params.step (params.nim:90-98) = add (:33-48) then scale (:61-66), the prox of
// minibatch_psgd.nim:119-121, and "grads <- 0" (:99) for the next minibatch, in one pass.
// tail = [gb, lossSum] (already all-reduced).  scal[0] accumulates the epoch's loss sum.
static __global__ void mbpsgd_step_kernel(double *P, double *gP, int64_t nP, double negEtaP, double rP, int reg,
                                   double lam, double *w, double *gw, int64_t d, double negEtaW, double rW,
                                   int fitLinear, double *b, double *tail, double negEtaB, double rB,
                                   int fitIntercept, double *scal) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  for (int64_t e = tid; e < nP; e += stride) {
    double p = P[e] + negEtaP * gP[e];
    p *= rP;
    if (reg == NIMFM_REG_L1) {  // softthreshold, regularizer/utils.nim:4-5
      const double m = fabs(p) - lam;
      p = (p > 0 ? 1.0 : (p < 0 ? -1.0 : 0.0)) * (m > 0.0 ? m : 0.0);
    }
    P[e] = p;
    gP[e] = 0.0;
  }
  if (fitLinear)
    for (int64_t e = tid; e < d; e += stride) {
      double v = w[e] + negEtaW * gw[e];
      w[e] = v * rW;
      gw[e] = 0.0;
    }
  else
    for (int64_t e = tid; e < d; e += stride) gw[e] = 0.0;
  if (tid == 0) {
    double bb = b[0];
    if (fitIntercept && fitLinear) bb += negEtaB * tail[0];  // params.nim:47 (quirk: needs grad.fitLinear)
    if (fitIntercept) bb *= rB;                              // params.nim:65-66
    b[0] = bb;
    scal[0] += tail[1];
    tail[0] = 0.0;
    tail[1] = 0.0;
  }
}

// The same step on ONE RANK'S FLAT SLICE [lo, hi) of the pools (multi-rank: reduce-scatter of the gradient pool
// -> this kernel on 1/N of the elements -> all-gather of the parameter pool).  par = [P | w | b, epochLoss],
// g = [gP | gw | gb, lossSum], both in the same flat element order; the slice may straddle the P / w / tail
// boundaries.  The gradient pool is cleared by the caller (every rank holds partial sums outside its slice).
static __global__ void mbpsgd_step_flat_kernel(double *par, const double *g, int64_t lo, int64_t hi, int64_t nP,
                                               int64_t d, double negEtaP, double rP, int reg, double lam,
                                               double negEtaW, double rW, int fitLinear, double negEtaB, double rB,
                                               int fitIntercept) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = lo + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < hi; e += stride) {
    if (e < nP) {
      double p = par[e] + negEtaP * g[e];
      p *= rP;
      if (reg == NIMFM_REG_L1) {
        const double m = fabs(p) - lam;
        p = (p > 0 ? 1.0 : (p < 0 ? -1.0 : 0.0)) * (m > 0.0 ? m : 0.0);
      }
      par[e] = p;
    } else if (e < nP + d) {
      if (fitLinear) par[e] = (par[e] + negEtaW * g[e]) * rW;
    } else if (e == nP + d) {
      double bb = par[e];
      if (fitIntercept && fitLinear) bb += negEtaB * g[e];   // params.nim:47
      if (fitIntercept) bb *= rB;                            // params.nim:65-66
      par[e] = bb;
    } else if (e == nP + d + 1) {
      par[e] += g[e];                                        // the epoch's loss sum (minibatch_psgd.nim:84,124)
    }
  }
}

// ------------------------------------------------------------------ MBPSGD lazy step (K3b)
// The dense step above moves all of P, w and the gradient buffer every minibatch; with the reference's
// default minibatch (25 641 rows of the Criteo shape) a minibatch touches ~1/5 of the features and the
// dense pass costs as much as the row kernel.  An untouched feature only shrinks: p <- p / (1 + eta_t beta).
// The lazy epoch applies that shrink when the feature is next touched: with cum[t] = prod_{s<t} r_s the
// pending factor of feature j is cum[t] * inv[j] (inv[j] = 1 / cum at j's last update); the row kernel
// folds it into x (fm_rows_stream.cuh), so the gradient it scatters is the true one times the same
// factor.  One flat kernel then updates the touched features only: their P rows and the per-feature state (w, inv,
// flag); its block 0 also folds the row kernel's partials into the intercept step and the epoch's loss sum, i.e.
// reduce_partials + add_tail + the tid == 0 branch of mbpsgd_step_kernel.  SB8 = 1 << shift.
// One pass, a warp per 32 consecutive features: ONE coalesced 32-byte read of their flags, a ballot, and only the
// touched features are visited -- their P rows by 2^shift lanes each (32 >> shift features side by side when a row
// is shorter than a warp), then w / inv / flag by the lanes that own them.  (Round 1 had an element-wise P kernel
// that looked a flag up per ELEMENT plus a second walk over the flags for the feature state: same results; the
// fused form is +16 % on 4 096-row minibatch SGD and even on C3's 25 641-row minibatches, where the touched rows'
// own traffic -- ~100 MB of scattered 128-byte rows -- is what the step costs.)
static __global__ void __launch_bounds__(256) mbpsgd_lazy_step_kernel(
    double *__restrict__ P, double *__restrict__ gP, int shift, int64_t dd, int64_t d, double *w, double *gw,
    uint8_t *flag, double2 *inv, double cumPt, double cumWt, double invPnext, double invWnext, double negEtaP, double rP,
    double aP, double negEtaW, double rW, double aW, int fitLinear, double *b, const double *partials,
    int64_t partialRows, double negEtaB, double rB, int fitIntercept, double *scal, double *violPart) {
  __shared__ double red[8];
  double viol = 0.0;
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nWarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int SB8 = 1 << shift;
  const int fpw = shift >= 5 ? 1 : (32 >> shift);          // features side by side in one pass over P
  const int sub = shift >= 5 ? 0 : (lane >> shift);
  const int el = shift >= 5 ? lane : (lane & (SB8 - 1));
  for (int64_t j0 = warp * 32; j0 < dd; j0 += nWarps * 32) {
    const int64_t j = j0 + lane;
    const bool on = j < dd && flag[j] != 0;
    const unsigned mask = __ballot_sync(0xffffffffu, on);
    if (!mask) continue;
    double2 iv = make_double2(1.0, 1.0);
    if (on) iv = inv[j];
    // ---- P rows of the touched features: p <- (aP p_eff - eta g_true) rP, g <- 0
    unsigned m = mask;
    while (m) {
      unsigned mm = m;                                      // this sub-group takes the sub-th set bit of m
      for (int i = 0; i < sub; i++) mm &= mm - 1;
      const int f = mm ? __ffs(mm) - 1 : -1;
      const double ivx = __shfl_sync(0xffffffffu, iv.x, f < 0 ? 0 : f);
      if (f >= 0) {
        const double fac = cumPt * ivx;
        const int64_t base = (j0 + f) << shift;
        for (int e = el; e < SB8; e += 32) {
          const double pe = P[base + e] * fac;
          const double p = (aP * pe + negEtaP * (gP[base + e] / fac)) * rP;
          viol += fabs(p - pe);
          P[base + e] = p;
          gP[base + e] = 0.0;
        }
      }
      for (int i = 0; i < fpw && m; i++) m &= m - 1;
    }
    // ---- per-feature state: w likewise, inv[j] <- 1 / cum[t+1], flag reset
    if (on) {
      if (j < d) {
        if (fitLinear) {
          const double we = w[j] * (cumWt * iv.y);
          const double v = (aW * we + negEtaW * (gw[j] / (cumPt * iv.x))) * rW;
          viol += fabs(v - we);
          w[j] = v;
        }
        gw[j] = 0.0;
      }
      inv[j] = make_double2(invPnext, invWnext);
      flag[j] = 0;
    }
  }
  if (blockIdx.x == 0) {
    double acc0 = 0.0, acc1 = 0.0;
    for (int64_t r = threadIdx.x; r < partialRows; r += 256) {
      acc0 += partials[r * 4 + 0];
      acc1 += partials[r * 4 + 1];
    }
    const double lossSum = block_sum(acc0, red);
    __syncthreads();
    const double gb = block_sum(acc1, red);
    if (threadIdx.x == 0) {
      double bb = b[0];
      if (violPart) {                                        // sgd.nim:225-228
        if (fitIntercept) {
          const double bn = rB * bb + negEtaB * gb;
          viol += fabs(bn - bb);
          bb = bn;
        }
      } else {
        if (fitIntercept && fitLinear) bb += negEtaB * gb;   // params.nim:47
        if (fitIntercept) bb *= rB;                          // params.nim:65-66
      }
      b[0] = bb;
      scal[0] += lossSum;
    }
    __syncthreads();
  }
  if (violPart) {
    viol = block_sum(viol, red);
    if (threadIdx.x == 0) {
      violPart[blockIdx.x * 4 + 0] = viol;
      violPart[blockIdx.x * 4 + 1] = 0.0;
      violPart[blockIdx.x * 4 + 2] = 0.0;
      violPart[blockIdx.x * 4 + 3] = 0.0;
    }
  }
}

// end of a lazy epoch: every feature receives the shrink it still owes (P here, w + the reset of inv below)
static __global__ void mbpsgd_lazy_flush_P_kernel(double *P, int shift, int64_t nP, const double2 *inv, double cumPT) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < nP; e += stride) P[e] *= cumPT * inv[e >> shift].x;
}
static __global__ void mbpsgd_lazy_flush_feat_kernel(double *w, int64_t d, int fitLinear, double2 *inv, int64_t dd,
                                                     double cumWT) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < dd; j += stride) {
    if (fitLinear && j < d) w[j] *= cumWT * inv[j].y;
    inv[j] = make_double2(1.0, 1.0);
  }
}

// ------------------------------------------------------------------ AdaGrad dense kernels (K5)
// A minibatch runs: count -> [all-reduce counts] -> refresh -> row kernel (reads P, scatters the
// deltas) -> [all-reduce deltas] -> scalar + apply.
//
// cnt[j] += number of rows of the batch that contain feature j (dummy features: every row).
// Columns of the dataset's hot table (present in >= 1/16 of the rows) are counted in shared memory and
// flushed once per block: 1 Mi Criteo-shaped rows put 1 Mi REDs on each of 13 addresses otherwise (4.3 ms
// of a 14 ms minibatch).  Counts are small integers held in doubles: exact in any order.
static __global__ void adagrad_count_kernel(const int32_t *indices, const int64_t *indptr, int64_t n, int64_t rowBegin,
                                            int64_t nRows, const int32_t *rowIdx, int64_t d, int nAug, double *cnt,
                                            const uint8_t *hotSlot, const int32_t *hotList, int nHot) {
  __shared__ int hotCnt[16];
  if (threadIdx.x < 16) hotCnt[threadIdx.x] = 0;
  __syncthreads();
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nWarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int lane = threadIdx.x & 31;
  for (int64_t q = warp; q < nRows; q += nWarps) {
    const int64_t r = rowIdx ? (int64_t)rowIdx[q] : (rowBegin + q) % n;
    for (int64_t e = indptr[r] + lane; e < indptr[r + 1]; e += 32) {
      const int32_t j = indices[e];
      const int slot = (hotSlot && nHot > 0) ? hotSlot[j] : 255;
      if (slot != 255) atomicAdd(&hotCnt[slot], 1);
      else atomicAdd(cnt + j, 1.0);
    }
  }
  __syncthreads();
  if ((int)threadIdx.x < nHot && hotCnt[threadIdx.x] > 0) atomicAdd(cnt + hotList[threadIdx.x], (double)hotCnt[threadIdx.x]);
  if (warp == 0 && lane < nAug) cnt[d + lane] += (double)nRows;   // augmentation: one dummy per row
}

// The two per-minibatch AdaGrad passes below visit ONLY the features the batch touches (cnt[j] != 0):
// (see the block-level scheme below); every touched feature's SB8 contiguous elements are handled by one warp.  Untouched features carry zero deltas by construction, so skipping them is
// exact; for FFM (nFields*k = 312 elements per feature, P = 2.5 GB) a dense pass per minibatch cost
// more than the row kernel itself.
//
// update() of adagrad.nim:87-110 for every feature the batch touches, done ONCE per feature:
// theta = -eta0*G/(eta0*t*reg + sqrt(N)); viol += cnt[j] * |P_old - theta| (the reference adds the
// same |P_old - theta| once per row containing j, and 0 for every later row of the batch -- with the
// snapshot semantics of the synchronous minibatch every incidence sees the pre-batch P).
// partials: [gridDim][4], column 3 = viol.
// Both passes: a block reads 256 counts (coalesced), lists its touched features in shared memory in index
// order, and its warps take them round-robin; a feature's SB8 elements are handled 4 x 32 at a time with
// all loads of a batch issued before the first is used (ncu on the first form -- 32 features per warp,
// one dependent round trip per 32 elements -- showed 12 ms per call at 4 % DRAM: pure load latency).
#define ADA_UNROLL 4
static __global__ void adagrad_refresh_kernel(double *P, const double *gsP, const double *gnP, int64_t dd, int SB8,
                                              const double *cnt, double *w, const double *gsw, const double *gnw,
                                              int64_t d, int fitLinear, double eta0, double tIt, double alpha,
                                              double beta, double *partials) {
  __shared__ double red[8];
  __shared__ int sList[256];
  __shared__ double sCnt[256];
  __shared__ int sN;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const double tmpP = eta0 * tIt * beta;
  const double denW = tIt * eta0 * alpha;
  double viol = 0.0;
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < dd; base += (int64_t)gridDim.x * blockDim.x) {
    const int64_t jm = base + threadIdx.x;
    const double cm = jm < dd ? cnt[jm] : 0.0;
    if (fitLinear && cm != 0.0 && jm < d) {
      const double wn = -eta0 * gsw[jm] / (denW + sqrt(gnw[jm]));   // fitLinearAdaGrad, fit_linear.nim:50-57
      viol += cm * fabs(w[jm] - wn);
      w[jm] = wn;
    }
    __syncthreads();
    if (threadIdx.x == 0) sN = 0;
    __syncthreads();
    // ordered compaction of this block's touched features (deterministic: warp order, then lane order)
    const unsigned mask = __ballot_sync(0xffffffffu, cm != 0.0);
    for (int ww = 0; ww < nw; ++ww) {
      if (wid == ww && cm != 0.0) {
        const int pos = sN + __popc(mask & ((1u << lane) - 1));
        sList[pos] = threadIdx.x;
        sCnt[pos] = cm;
      }
      __syncthreads();
      if (threadIdx.x == ww * 32) sN += __popc(mask);
      __syncthreads();
    }
    const int nT = sN;
    for (int t = wid; t < nT; t += nw) {
      const double c = sCnt[t];
      const int64_t e0 = (base + sList[t]) * SB8;
      for (int eb = 0; eb < SB8; eb += 32 * ADA_UNROLL) {
        double g[ADA_UNROLL], nn[ADA_UNROLL], p[ADA_UNROLL];
#pragma unroll
        for (int i = 0; i < ADA_UNROLL; ++i) {
          const int e = eb + lane + 32 * i;
          const bool ok = e < SB8;
          g[i] = ok ? gsP[e0 + e] : 0.0;
          nn[i] = ok ? gnP[e0 + e] : 1.0;
          p[i] = ok ? P[e0 + e] : 0.0;
        }
#pragma unroll
        for (int i = 0; i < ADA_UNROLL; ++i) {
          const int e = eb + lane + 32 * i;
          if (e < SB8) {
            const double pn = -(eta0 * g[i]) / (tmpP + sqrt(nn[i]));
            viol += c * fabs(p[i] - pn);
            P[e0 + e] = pn;
          }
        }
      }
    }
  }
  viol = block_sum(viol, red);
  if (threadIdx.x == 0) {
    partials[blockIdx.x * 4 + 0] = 0.0;
    partials[blockIdx.x * 4 + 1] = 0.0;
    partials[blockIdx.x * 4 + 2] = 0.0;
    partials[blockIdx.x * 4 + 3] = viol;
  }
}

// updateG() of adagrad.nim:113-134 for the touched features: g_sum += dGs, g_norm += dGn, deltas and
// counts cleared.
static __global__ void adagrad_apply_kernel(double *gsP, double *gnP, double *dGsP, double *dGnP, int64_t nP,
                                            double *gsw, double *gnw, double *dGsw, double *dGnw, int64_t d,
                                            int fitLinear, double *cnt, int64_t dd) {
  __shared__ int sList[256];
  __shared__ int sN;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int SB8 = (int)(nP / dd);
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < dd; base += (int64_t)gridDim.x * blockDim.x) {
    const int64_t jm = base + threadIdx.x;
    const double cm = jm < dd ? cnt[jm] : 0.0;
    if (cm != 0.0) {
      if (jm < d) {
        if (fitLinear) {
          gsw[jm] += dGsw[jm];
          gnw[jm] += dGnw[jm];
        }
        dGsw[jm] = 0.0;
        dGnw[jm] = 0.0;
      }
      cnt[jm] = 0.0;
    }
    __syncthreads();
    if (threadIdx.x == 0) sN = 0;
    __syncthreads();
    if (cm != 0.0) sList[atomicAdd(&sN, 1)] = threadIdx.x;   // order is irrelevant here: features are independent
    __syncthreads();
    const int nT = sN;
    for (int t = wid; t < nT; t += nw) {
      const int64_t e0 = (base + sList[t]) * SB8;
      for (int eb = 0; eb < SB8; eb += 32 * ADA_UNROLL) {
        double gs[ADA_UNROLL], gn[ADA_UNROLL], ds[ADA_UNROLL], dn[ADA_UNROLL];
#pragma unroll
        for (int i = 0; i < ADA_UNROLL; ++i) {
          const int e = eb + lane + 32 * i;
          const bool ok = e < SB8;
          gs[i] = ok ? gsP[e0 + e] : 0.0;
          gn[i] = ok ? gnP[e0 + e] : 0.0;
          ds[i] = ok ? dGsP[e0 + e] : 0.0;
          dn[i] = ok ? dGnP[e0 + e] : 0.0;
        }
#pragma unroll
        for (int i = 0; i < ADA_UNROLL; ++i) {
          const int e = eb + lane + 32 * i;
          if (e < SB8) {
            gsP[e0 + e] = gs[i] + ds[i];
            gnP[e0 + e] = gn[i] + dn[i];
            dGsP[e0 + e] = 0.0;
            dGnP[e0 + e] = 0.0;
          }
        }
      }
    }
  }
}
// intercept part of update()/updateG() (adagrad.nim:101-105,126-128) + epoch accumulators.
// part = [loss, sum dL, sum dL^2, -] of the batch (all-reduced); violRefresh = this rank's viol of the
// refresh pass (identical on every rank: counts are all-reduced first); scal = [lossEpoch, violEpoch]
static __global__ void adagrad_scalar_kernel(double *b, double *adaScal, const double *part, const double *violRefresh,
                                      double *scal, int fitIntercept, double eta0, double tIt, double alpha0,
                                      int first) {
  double viol = first ? 0.0 : violRefresh[3];
  if (fitIntercept) {
    if (!first) {
      const double old = b[0];
      const double den = sqrt(adaScal[1]) + eta0 * tIt * alpha0;
      const double nb = -eta0 * adaScal[0] / den;
      viol += fabs(old - nb);
      b[0] = nb;
    }
    adaScal[0] += part[1];
    adaScal[1] += part[2];
  }
  scal[0] += part[0];
  scal[1] += viol;
}

// coef_i = dloss(y_i, yhat_i) / mb in place of yhat (a forward kernel's output), and the loss / sum coef / sum dL^2
// partials per block: their order depends on nRows and the grid only, not on the forward kernel (the column routes)
static __global__ void dloss_coef_kernel(double *yhatCoef, const double *y, int64_t rowBegin, int64_t nRows, int loss,
                                         double thr, double mb, double *partials) {
  __shared__ double red[8];
  double l = 0.0, c = 0.0, d2 = 0.0;
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nRows; q += (int64_t)gridDim.x * blockDim.x) {
    const double yi = y[rowBegin + q], yh = yhatCoef[q];
    const double dL = dev_dloss(loss, thr, yi, yh);
    l += dev_loss(loss, thr, yi, yh);
    c += dL / mb;
    d2 += dL * dL;
    yhatCoef[q] = dL / mb;
  }
  l = block_sum(l, red);
  __syncthreads();
  c = block_sum(c, red);
  __syncthreads();
  d2 = block_sum(d2, red);
  if (threadIdx.x == 0) {
    partials[blockIdx.x * 4 + 0] = l;
    partials[blockIdx.x * 4 + 1] = c;
    partials[blockIdx.x * 4 + 2] = d2;
    partials[blockIdx.x * 4 + 3] = 0.0;
  }
}

// the intercept every row of an AdaGrad minibatch sees (adagrad.nim:101-105), written to *out for a forward pass that
// reads its intercept from memory: the same expression as the AdaGrad row kernels' prologue (fm_rows.cuh, ffm.cu)
static __global__ void adagrad_bias_kernel(double *out, const double *b, const double *adaScal, int fitIntercept,
                                           int first, double eta0, double tIt, double alpha0) {
  double bias = b[0];
  if (!first && fitIntercept) {
    const double den = sqrt(adaScal[1]) + eta0 * tIt * alpha0;
    bias = -eta0 * adaScal[0] / den;
  }
  *out = bias;
}
// AdaGrad.finalize (adagrad.nim:65-84)
static __global__ void adagrad_finalize_kernel(double *P, const double *gsP, const double *gnP, int64_t nP, double *w,
                                        const double *gsw, const double *gnw, int64_t d, int fitLinear,
                                        double *b, const double *adaScal, int fitIntercept, double eta0,
                                        double tIt, double alpha0, double alpha, double beta) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const double denP = eta0 * tIt * beta;
  for (int64_t e = tid; e < nP; e += stride) P[e] = (-eta0 * gsP[e]) / (denP + sqrt(gnP[e]));
  if (fitLinear) {
    const double denW = eta0 * tIt * alpha;
    for (int64_t j = tid; j < d; j += stride) w[j] = (-eta0 * gsw[j]) / (denW + sqrt(gnw[j]));
  }
  if (tid == 0 && fitIntercept) {
    const double den = sqrt(adaScal[1]) + eta0 * tIt * alpha0;
    b[0] = -eta0 * adaScal[0] / den;
  }
}
static __global__ void fill_kernel(double *p, int64_t n, double v) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) p[e] = v;
}


// tail[0] (gb) += sum coef, tail[1] (loss) += sum loss; red4 = reduce_partials output
static __global__ void add_tail_kernel(double *tail, const double *red4) {
  tail[0] += red4[1];
  tail[1] += red4[0];
}
