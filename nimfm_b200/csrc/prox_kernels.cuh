// prox_kernels.cuh -- proximal operators of MBPSGD on the device (SURVEY 8f.1; called after the dense
// step exactly where minibatch_psgd.nim:119-121 calls reg.prox(params.P[order], lam, degree-order)):
//   L21.prox                     regularizer/l21.nim:25-35       one vector per (feature, order), k elements
//   SquaredL12.prox transpose=f  regularizer/squaredl12.nim:157-159  same vectors
//   SquaredL12.prox transpose=t  regularizer/squaredl12.nim:147-156  one vector per (order, component)
//                                                                    over ALL d+nAug features
// Device layout P[j][o][s]: a (feature, order) vector is k contiguous doubles; an (order, component)
// vector is the column c = o*k+s with stride SB8 = nOrders*k.
//
// proxSquaredL12 (squaredl12.nim:16-64) finds, by randomised selection, theta = the number of
// elements with |p_i| > tau where tau = 2*lam*S and S = sum_{|p_i| > tau} |p_i| / (1 + 2*lam*theta),
// then soft-thresholds by tau.  That fixed point is unique, and the pivot order does not change it, so
// the device computes it with Michelot's iteration: start from all elements, recompute tau from the
// active set {|p| > tau}, repeat until the set stops shrinking (tau only grows, each pass is one
// coalesced sweep with fixed-order reductions).  S is then formed exactly as the reference forms it.
// The iteration stops at the first pass whose count does not decrease and keeps the tau that pass took
// as input.  Stopping only on an equal count cycles in floating point when an element sits at the
// threshold of the others: the set with it rounds tau up to it (it drops out), the set without it rounds
// tau one ulp below it (it comes back), and the counts alternate n+1, n, n+1, ... for ever.
#pragma once
#include "common.cuh"

#define NIMFM_PROX_MAXE 4   // a (feature, order) vector may hold up to 32*MAXE components

// ------------------------------------------------------------------ row-wise: L21 / SquaredL12(transpose=false)
static __global__ void prox_rows_kernel(double *P, int64_t nRows, int k, double lam, int kind) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nWarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp; r < nRows; r += nWarps) {
    double *row = P + r * k;
    double p[NIMFM_PROX_MAXE];
#pragma unroll
    for (int i = 0; i < NIMFM_PROX_MAXE; ++i) p[i] = (lane + 32 * i < k) ? row[lane + 32 * i] : 0.0;
    if (kind == NIMFM_REG_L21) {
      double ss = 0.0;
#pragma unroll
      for (int i = 0; i < NIMFM_PROX_MAXE; ++i) ss += p[i] * p[i];
      const double nrm = sqrt(warp_sum(ss));
      const double f = nrm > lam ? 1.0 - lam / nrm : 0.0;         // l21.nim:27-29
#pragma unroll
      for (int i = 0; i < NIMFM_PROX_MAXE; ++i)
        if (lane + 32 * i < k) row[lane + 32 * i] = nrm > lam ? p[i] * f : 0.0;
    } else {
      double tau = -1.0, prevCnt = INFINITY;
      for (int iter = 0; iter < 4096; ++iter) {   // at most k + 2 passes: the count decreases until the last
        double cnt = 0.0, sum = 0.0;
#pragma unroll
        for (int i = 0; i < NIMFM_PROX_MAXE; ++i) {
          const double a = fabs(p[i]);
          if (lane + 32 * i < k && a > tau) { cnt += 1.0; sum += a; }
        }
        cnt = warp_sum(cnt);
        sum = warp_sum(sum);
        if (cnt >= prevCnt) break;                                 // keep the tau of the smaller set
        prevCnt = cnt;
        const double S = sum / (1.0 + 2.0 * lam * cnt);           // squaredl12.nim:67
        tau = 2 * lam * S;
      }
#pragma unroll
      for (int i = 0; i < NIMFM_PROX_MAXE; ++i)
        if (lane + 32 * i < k) {
          const double m = fabs(p[i]) - tau;
          row[lane + 32 * i] = (p[i] > 0 ? 1.0 : (p[i] < 0 ? -1.0 : 0.0)) * (m > 0.0 ? m : 0.0);
        }
    }
  }
}

// ------------------------------------------------------------------ column-wise: SquaredL12(transpose=true)
// state: [tau (SB8) | prevCnt (SB8) | settled (SB8) | done flag].  A column is settled by the first pass whose
// count does not decrease; from then on its tau stays put while the other columns iterate.
// One sweep: per column c, count and sum of |P[j][c]| > tau[c] over this block's features, written as
// partials[block][c][2].  blockDim.x = R * SB8: thread -> (feature-in-block r, column c).
static __global__ void sql12_pass_kernel(const double *P, int64_t dd, int SB8, int R, const double *state,
                                         double *partials) {
  extern __shared__ double sh[];   // [blockDim.x][2]
  const double *tau = state;
  if (state[3 * SB8] != 0.0) return;   // converged: nothing left to do
  const int c = threadIdx.x % SB8, rr = threadIdx.x / SB8;
  const double t = tau[c];
  double cnt = 0.0, sum = 0.0;
  for (int64_t j = (int64_t)blockIdx.x * R + rr; j < dd; j += (int64_t)gridDim.x * R) {
    const double a = fabs(P[j * SB8 + c]);
    if (a > t) { cnt += 1.0; sum += a; }
  }
  sh[2 * threadIdx.x] = cnt;
  sh[2 * threadIdx.x + 1] = sum;
  __syncthreads();
  if (rr == 0) {
    for (int r = 1; r < R; ++r) {
      cnt += sh[2 * (r * SB8 + c)];
      sum += sh[2 * (r * SB8 + c) + 1];
    }
    partials[((int64_t)blockIdx.x * SB8 + c) * 2] = cnt;
    partials[((int64_t)blockIdx.x * SB8 + c) * 2 + 1] = sum;
  }
}

// one block: fixed-order sum of the partials, new tau per unsettled column, convergence flag
static __global__ void sql12_update_kernel(const double *partials, int nBlocks, int SB8, double lam, double *state) {
  double *tau = state, *prevCnt = state + SB8, *settled = state + 2 * SB8, *done = state + 3 * SB8;
  if (*done != 0.0) return;
  int conv = 1;
  for (int c = threadIdx.x; c < SB8; c += blockDim.x) {
    if (settled[c] != 0.0) continue;
    double cnt = 0.0, sum = 0.0;
    for (int b = 0; b < nBlocks; ++b) {
      cnt += partials[((int64_t)b * SB8 + c) * 2];
      sum += partials[((int64_t)b * SB8 + c) * 2 + 1];
    }
    if (cnt >= prevCnt[c]) {                                      // keep the tau of the smaller set
      settled[c] = 1.0;
      continue;
    }
    conv = 0;
    prevCnt[c] = cnt;
    const double S = sum / (1.0 + 2.0 * lam * cnt);               // squaredl12.nim:67
    tau[c] = 2 * lam * S;                                         // the threshold of :69
  }
  const int all = __syncthreads_and(conv);
  if (threadIdx.x == 0 && all) *done = 1.0;
}

static __global__ void sql12_apply_kernel(double *P, int64_t dd, int SB8, int R, const double *state) {
  const int c = threadIdx.x % SB8, rr = threadIdx.x / SB8;
  const double t = state[c];
  for (int64_t j = (int64_t)blockIdx.x * R + rr; j < dd; j += (int64_t)gridDim.x * R) {
    const double p = P[j * SB8 + c];
    const double m = fabs(p) - t;
    P[j * SB8 + c] = (p > 0 ? 1.0 : (p < 0 ? -1.0 : 0.0)) * (m > 0.0 ? m : 0.0);   // softthreshold, utils.nim:4-5
  }
}

static __global__ void sql12_init_kernel(double *state, int SB8) {
  for (int c = threadIdx.x; c < SB8; c += blockDim.x) {
    state[c] = -1.0;             // tau: every element is active in the first pass
    state[SB8 + c] = INFINITY;   // prevCnt: the first pass never stops
    state[2 * SB8 + c] = 0.0;
  }
  if (threadIdx.x == 0) state[3 * SB8] = 0.0;
}
