// psgd.cu -- proximal SGD for FM (optimizer/psgd.nim:76-215), SURVEY 8f.2.
//
// PSGD is strictly sequential per sample, like SGD ("replicas only" for multi-GPU).  Two device routes:
//  * L1 / L21 (regularizer/l1.nim:84-136, l21.nim:36-112): the reference keeps the parameters of
//    untouched features stale and catches them up lazily (a global scaling / accumulated threshold and
//    the per-feature values they had at the last touch).  That bookkeeping is NOT algebraically equal to
//    an eager prox per step (e.g. l21.nim:86 accumulates eta*scaling with the pre-update scaling), so it
//    is reproduced literally: ONE persistent thread block runs the sample loop with the row's P slice
//    staged in shared memory (as sgd_fm_staged_kernel), applying lazyUpdate on the way in, the
//    regulariser's step() in place, and updateCacheSGD / resetCacheSGD after it.
//  * SquaredL12 (squaredl12.nim:199-230) is dense in the reference too ("sparsity is not leveraged"):
//    every sample updates ALL parameters and runs the full prox.  Here: row kernel on the one sample
//    (K2, coef = dloss) -> dense step kernel -> the MBPSGD prox kernels (prox_kernels.cuh).
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>

#include "dense_kernels.cuh"

#define PSGD_THREADS 256

extern "C" {   // library-internal helpers defined in fm_api.cu (inside its extern "C" block)
int nimfm_fm_loss_grad_one_row(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, int loss, double thr,
                               int64_t row);
int nimfm_fm_apply_prox(nimfm_ctx *ctx, nimfm_fm *fm, int reg, double lam);
}

__device__ __forceinline__ double psgd_eta(int sched, double eta0, double power, double reg, int64_t it) {
  switch (sched) {  // getEta, sgd.nim:60-69
    case NIMFM_SCHED_CONSTANT: return eta0;
    case NIMFM_SCHED_OPTIMAL: return eta0 / pow(1.0 + eta0 * reg * (double)it, power);
    case NIMFM_SCHED_INVSCALING: return eta0 / pow((double)it, power);
    default: return 1.0 / (reg * (double)it);
  }
}
static double host_eta(int sched, double eta0, double power, double reg, int64_t it) {
  switch (sched) {
    case NIMFM_SCHED_CONSTANT: return eta0;
    case NIMFM_SCHED_OPTIMAL: return eta0 / pow(1.0 + eta0 * reg * (double)it, power);
    case NIMFM_SCHED_INVSCALING: return eta0 / pow((double)it, power);
    default: return 1.0 / (reg * (double)it);
  }
}

__device__ __forceinline__ double psgd_soft(double x, double a) {   // softthreshold, regularizer/utils.nim:4-5
  const double m = fabs(x) - a;
  return (x > 0 ? 1.0 : (x < 0 ? -1.0 : 0.0)) * (m > 0.0 ? m : 0.0);
}

struct PsgdArgs {
  const double *data;
  const int32_t *indices;
  const int64_t *indptr;
  const double *y;
  const int32_t *perm;
  int64_t nRows, d, dd;
  int degree, k, nOrders, nAug;
  int fitLinear, fitIntercept;
  double *P, *w, *b;
  double *regScalings, *regThresholds, *scalingsW;   // [dd], [dd], [d]
  double *scal;                                      // [reg scaling, reg threshold, scaling_w, loss sum]
  nimfm_psgd_cfg cfg;
  int64_t it0;
  int zmax;
  int profile;   // NIMFM_PSGD_PROFILE: print the pipelined kernel's cycles per phase (debug)
};

// L21.prox of the k-vector at v (l21.nim:25-29) by one warp; every lane of the warp must call
__device__ __forceinline__ void psgd_l21_prox_warp(double *v, int k, double lam, double post) {
  const int lane = threadIdx.x & 31;
  double ss = 0.0;
  for (int s = lane; s < k; s += 32) ss += v[s] * v[s];
  const double nrm = sqrt(warp_sum(ss));
  const double f = nrm > lam ? 1.0 - lam / nrm : 0.0;
  for (int s = lane; s < k; s += 32) {
    double p = nrm > lam ? v[s] * f : 0.0;
    v[s] = p * post;
  }
}

// the same prox for up to EIGHT vectors of k <= 32 components per warp at a time (v0, v0+nw, ...), as STRAIGHT-LINE
// code: lane <-> component, the element stays in a register from the norm to the write-back.  This single block is
// bound by the latency of dependent instructions (~5 cycles each, 9 per FP64 operation, ~100 per sqrt or divide),
// and the generic form above costs ~1000 of them per vector in loop and branch overhead (measured: 9 000 cycles per
// prox round of a 39-nonzero row, more than the rest of the sample).  Here the eight sums are reduced with
// interleaved butterflies (every lane ends up with all of them), LANE c runs the sqrt / divide of vector c, and the
// factors are broadcast back: one sqrt -> divide chain per call.  lamTab / postTab are indexed by v / NO when
// non-null (the lazy catch-up), else lamC / 1.0 (the step's prox).  Every lane of the warp must call.
__device__ __forceinline__ void psgd_l21_prox_warp_x8(double *sP, int v0, int nw, int nv, int k, int NO,
                                                      const double *lamTab, const double *postTab, double lamC) {
  const int lane = threadIdx.x & 31;
  const bool inK = lane < k;
  double xr[8], ss[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int v = v0 + c * nw;
    xr[c] = (v < nv && inK) ? sP[(size_t)v * k + lane] : 0.0;
    ss[c] = xr[c] * xr[c];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
#pragma unroll
    for (int c = 0; c < 8; ++c) ss[c] += __shfl_xor_sync(0xffffffffu, ss[c], o);
  double mine = ss[0];
#pragma unroll
  for (int c = 1; c < 8; ++c)
    if (lane == c) mine = ss[c];
  const int vMine = v0 + lane * nw;
  double f = 0.0, post = 1.0;
  if (lane < 8 && vMine < nv) {
    const double lam = lamTab ? lamTab[vMine / NO] : lamC;
    if (postTab) post = postTab[vMine / NO];
    const double nrm = sqrt(mine);
    f = nrm > lam ? 1.0 - lam / nrm : -1.0;   // -1: the vector is zeroed (a factor is never negative)
  }
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int v = v0 + c * nw;
    const double fc = __shfl_sync(0xffffffffu, f, c), pc = __shfl_sync(0xffffffffu, post, c);
    const double p = fc >= 0.0 ? xr[c] * fc : 0.0;
    if (v < nv && inK) sP[(size_t)v * k + lane] = p * pc;
  }
}

// dynamic smem: sP[zmax*SB8] | sX | sW | sSc | sTh (zmax doubles each) | sJ[zmax] (int64)
__global__ void __launch_bounds__(PSGD_THREADS, 1) psgd_lazy_kernel(const PsgdArgs a) {
  extern __shared__ __align__(16) unsigned char psgd_smem[];
  __shared__ double red[PSGD_THREADS / 32];
  __shared__ double sh[8];   // 0 yhat, 1 reg scaling, 2 reg threshold, 3 scaling_w, 4 dL
  const int k = a.k, NO = a.nOrders, SB8 = NO * k, zmax = a.zmax;
  double *sP = reinterpret_cast<double *>(psgd_smem);
  double *sX = sP + (size_t)zmax * SB8;
  double *sW = sX + zmax;
  double *sSc = sW + zmax;
  double *sTh = sSc + zmax;
  int64_t *sJ = reinterpret_cast<int64_t *>(sTh + zmax);
  const int tid = threadIdx.x, nth = blockDim.x, wid = tid >> 5, nw = nth >> 5;
  const bool isL1 = a.cfg.reg == NIMFM_REG_L1;
  const double alpha0 = a.cfg.alpha0, alpha = a.cfg.alpha, beta = a.cfg.beta, gamma = a.cfg.gamma;
  double lossAcc = 0.0;
  if (tid == 0) {
    sh[1] = a.scal[0];
    sh[2] = a.scal[1];
    sh[3] = a.scal[2];
  }
  __syncthreads();
  for (int64_t q = 0; q < a.nRows; ++q) {
    const int64_t i = a.perm ? (int64_t)a.perm[q] : q;
    const int64_t it = a.it0 + q;
    const int64_t rb = a.indptr[i];
    const int zReal = (int)(a.indptr[i + 1] - rb);
    const int z = zReal + a.nAug;
    const double rSc = sh[1], rTh = sh[2], scW = sh[3];
    // ---- records + the lazy factors of every row feature incl. dummies (psgd.nim:121-127)
    for (int u = tid; u < z; u += nth) {
      const int64_t j = u < zReal ? (int64_t)a.indices[rb + u] : a.d + (u - zReal);
      sJ[u] = j;
      sX[u] = u < zReal ? a.data[rb + u] : 1.0;
      sW[u] = u < zReal ? a.w[j] * (scW / a.scalingsW[j]) : 0.0;       // sfm.w[j] *= scaling_w / scalings_w[j]
      const double sj = a.regScalings[j], tj = a.regThresholds[j];
      sSc[u] = rSc / sj;
      sTh[u] = isL1 ? gamma * rSc * (rTh - tj)                         // l1.nim:89-90
                    : ((rTh - tj) / sj) * gamma;                       // l21.nim:62-63
    }
    __syncthreads();
    for (int e = tid; e < z * SB8; e += nth) {
      const int u = e / SB8, off = e - u * SB8;
      double p = a.P[sJ[u] * SB8 + off];
      if (isL1) {                                                      // l1.nim:86-90
        p *= sSc[u];
        p = psgd_soft(p, sTh[u]);
      }
      sP[e] = p;
    }
    __syncthreads();
    if (!isL1) {                                                       // l21.nim:60-65: prox, then scale
      for (int v = wid; v < z * NO; v += nw) {
        const int u = v / NO;
        psgd_l21_prox_warp(sP + (size_t)v * k, k, sTh[u], sSc[u]);     // vector (u, o) = sP[u*SB8 + o*k ..]
      }
      __syncthreads();
    }
    // ---- predictWithGrad forward (thread <-> (order, component)); A stays in registers
    double part = 0.0;
    for (int u = tid; u < zReal; u += nth) part += sW[u] * sX[u];
    AnovaState A;
    const int os = tid;
    const int o = os < SB8 ? os / k : 0, sc = os - o * k;
    const int M = a.degree - o;
    if (os < SB8) {
      part += anova_forward_smem(A, M, sP + o * k + sc, SB8, sX, z);
    }
    double yhat = block_sum(part, red);
    if (tid == 0) {
      yhat += a.b[0];
      sh[0] = yhat;
      const double yi = a.y[i];
      lossAcc += dev_loss(a.cfg.loss, a.cfg.huberThreshold, yi, yhat);
      sh[4] = dev_dloss(a.cfg.loss, a.cfg.huberThreshold, yi, yhat);
    }
    __syncthreads();
    const double dL = sh[4];
    const double etaW = psgd_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha, it);
    const double etaP = psgd_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, beta, it);
    const double etaS = etaP / (1.0 + etaP * beta);                     // psgd.nim:134
    // ---- reg.step (l1.nim:127-136 / l21.nim:102-112)
    if (os < SB8) {
      for (int u = 0; u < z; u++) {
        const double x = sX[u];
        const int e = u * SB8 + o * k + sc;
        const double p = sP[e];
        double g;
        if (M == 2) g = x * (A[1] - p * x);
        else {
          g = anova_deriv(A, M, x, p);
        }
        const double upd = etaS * (dL * g + beta * p);
        sP[e] = isL1 ? psgd_soft(p - upd, gamma * etaS) : p - upd;
      }
    }
    __syncthreads();
    if (!isL1) {
      for (int v = wid; v < z * NO; v += nw) psgd_l21_prox_warp(sP + (size_t)v * k, k, etaS * gamma, 1.0);
      __syncthreads();
    }
    for (int e = tid; e < z * SB8; e += nth) {
      const int u = e / SB8, off = e - u * SB8;
      a.P[sJ[u] * SB8 + off] = sP[e];
    }
    // ---- reg.updateCacheSGD (l1.nim:106-113 / l21.nim:84-90), w, intercept, caches
    double nSc, nTh;
    if (isL1) {
      nTh = rTh + etaS / rSc;
      nSc = rSc * (1 - etaS * beta);
    } else {
      nTh = rTh + etaP * rSc;
      nSc = rSc / (1 + etaP * beta);
    }
    const double nScW = scW / (1.0 + etaW * alpha);                     // psgd.nim:153
    for (int u = tid; u < z; u += nth) {
      const int64_t j = sJ[u];
      a.regScalings[j] = nSc;
      a.regThresholds[j] = nTh;
      if (u < zReal) {
        if (a.fitLinear) {                                              // fitLinearSGD with eta_w/(1+eta_w*alpha)
          const double eta = etaW / (1.0 + etaW * alpha);
          a.w[j] = sW[u] - eta * (dL * sX[u] + alpha * sW[u]);
        }
        a.scalingsW[j] = nScW;
      }
    }
    if (tid == 0) {
      if (a.fitIntercept) {                                             // psgd.nim:146-148
        const double e0 = psgd_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha0, it);
        const double upd = e0 * (dL + alpha0 * a.b[0]);
        a.b[0] -= upd / (1.0 + e0 * alpha0);
      }
      sh[1] = nSc;
      sh[2] = nTh;
      sh[3] = nScW;
    }
    __syncthreads();
    // ---- resets against underflow (psgd.nim:158-163; l1.nim:116-124 and l21.nim:93-104 as written)
    if (a.fitLinear && nScW < 1e-9) {
      for (int64_t j = tid; j < a.d; j += nth) {
        double v = a.w[j] * nScW;
        a.w[j] = v / a.scalingsW[j];
        a.scalingsW[j] = 1.0;
      }
      __syncthreads();
      if (tid == 0) sh[3] = 1.0;
      __syncthreads();
    }
    if (nSc < 1e-8) {
      if (isL1) {
        for (int64_t e = tid; e < a.dd * SB8; e += nth) {
          const int64_t j = e / SB8;
          double p = a.P[e] / a.regScalings[j];
          p = psgd_soft(p, gamma * nTh - a.regThresholds[j]);
          a.P[e] = p * nTh;
        }
      } else {
        for (int64_t v = wid; v < a.dd * NO; v += nw) {
          const int64_t j = v / NO;
          const double thr = (nTh - a.regThresholds[j]) / a.regScalings[j];
          psgd_l21_prox_warp(a.P + v * k, k, thr * gamma, nSc / a.regScalings[j]);
        }
      }
      __syncthreads();
      for (int64_t j = tid; j < a.dd; j += nth) {
        a.regScalings[j] = 1.0;
        a.regThresholds[j] = 0.0;
      }
      if (tid == 0) {
        sh[1] = 1.0;
        sh[2] = 0.0;
      }
      __syncthreads();
    }
  }
  lossAcc = block_sum(lossAcc, red);
  if (tid == 0) {
    a.scal[0] = sh[1];
    a.scal[1] = sh[2];
    a.scal[2] = sh[3];
    a.scal[3] = lossAcc;
  }
}

// The same loop PIPELINED (as sgd_fm_pipe_kernel / adagrad_fm_pipe_kernel): the read-only CSR side of the dependent
// load chain (permutation -> row pointer / target -> indices / values) is fetched one to three samples ahead by the
// last warp; the row's P slice, w and the lazy caches -- what the previous sample may have changed -- are ONE round
// of independent loads held in registers until the lazy factors are known; the step is element <-> thread on the
// whole block and, for L1, goes straight to global memory.  Rows of at most 64 nonzeros, z*SB8 <= PIPE_R*threads.
// dynamic smem: sP[zmax*SB8] | sA[SB8*(MAXDEG+1)] | sX[2][zmax] | sW | sSc | sTh (zmax each) | sJ[2][zmax] (int32) | sOrd[SB8]
#define PSGD_PIPE_THREADS 512
#define PSGD_PIPE_R 12
struct PsgdPipeMeta {
  int64_t i, rb;
  double y;
  int z;
};

__global__ void __launch_bounds__(PSGD_PIPE_THREADS, 1) psgd_lazy_pipe_kernel(const PsgdArgs a) {
  extern __shared__ __align__(16) unsigned char psgd_smem[];
  __shared__ double red[PSGD_PIPE_THREADS / 32];
  __shared__ double sh[8];   // 1 reg scaling, 2 reg threshold, 3 scaling_w, 4 dL
  __shared__ PsgdPipeMeta meta[4];
  __shared__ double sEta[8];   // [q & 1][eta_w, eta_P, eta_0, -]
  const int k = a.k, NO = a.nOrders, SB8 = NO * k, zmax = a.zmax, AST = NIMFM_MAX_DEGREE + 1;
  double *sP = reinterpret_cast<double *>(psgd_smem);
  double *sA = sP + (size_t)zmax * SB8;
  double *sXb = sA + (size_t)SB8 * AST;
  double *sW = sXb + 2 * (size_t)zmax;
  double *sSc = sW + zmax;
  double *sTh = sSc + zmax;
  int32_t *sJb = reinterpret_cast<int32_t *>(sTh + zmax);
  const int tid = threadIdx.x, nth = blockDim.x, wid = tid >> 5, nw = nth >> 5, lastWarp0 = nth - 32;
  const bool isL1 = a.cfg.reg == NIMFM_REG_L1;
  const double alpha0 = a.cfg.alpha0, alpha = a.cfg.alpha, beta = a.cfg.beta, gamma = a.cfg.gamma;
  double lossAcc = 0.0;
  long long prof[7] = {0, 0, 0, 0, 0, 0, 0};
  ElemWalk walk0;
  walk0.start(tid, nth, SB8);
  signed char *sOrd = reinterpret_cast<signed char *>(sJb + 2 * zmax);   // [SB8] ANOVA order of (order, component) slot
  for (int os = tid; os < SB8; os += nth) sOrd[os] = (signed char)(a.degree - os / k);
  if (tid == 32) {
    sEta[0] = psgd_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha, a.it0);
    sEta[1] = psgd_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, beta, a.it0);
    sEta[2] = psgd_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha0, a.it0);
  }
  if (tid == 0) {
    sh[1] = a.scal[0];
    sh[2] = a.scal[1];
    sh[3] = a.scal[2];
    for (int64_t q = 0; q < 3 && q < a.nRows; ++q) {
      PsgdPipeMeta m;
      m.i = a.perm ? (int64_t)a.perm[q] : q;
      m.rb = 0; m.z = 0; m.y = 0.0;
      if (q < 2) {
        m.rb = a.indptr[m.i];
        m.z = (int)(a.indptr[m.i + 1] - m.rb);
        m.y = a.y[m.i];
      }
      meta[q & 3] = m;
    }
  }
  __syncthreads();
  if (tid >= lastWarp0 && a.nRows > 0) {
    const PsgdPipeMeta m = meta[0];
    for (int u = tid - lastWarp0; u < m.z + a.nAug; u += 32) {
      sJb[u] = u < m.z ? a.indices[m.rb + u] : (int32_t)(a.d + (u - m.z));
      sXb[u] = u < m.z ? a.data[m.rb + u] : 1.0;
    }
  }
  __syncthreads();
  for (int64_t q = 0; q < a.nRows; ++q) {
    const int64_t it = a.it0 + q;
    const PsgdPipeMeta m = meta[q & 3];
    const int zReal = m.z, z = zReal + a.nAug;
    const int32_t *J = sJb + (q & 1) * zmax;
    const double *X = sXb + (q & 1) * zmax;
    const double rSc = sh[1], rTh = sh[2], scW = sh[3];
    // ---- fetch ahead (registers now, shared memory at the end of the iteration)
    int64_t pfI = 0, pfRb = 0, pfRe = 0;
    double pfY = 0.0, pfX0 = 0.0, pfX1 = 0.0;
    int32_t pfJ0 = 0, pfJ1 = 0;
    if (tid == nth - 1) {
      if (q + 3 < a.nRows) pfI = a.perm ? (int64_t)a.perm[q + 3] : q + 3;
      if (q + 2 < a.nRows) {
        const int64_t i2 = meta[(q + 2) & 3].i;
        pfRb = a.indptr[i2];
        pfRe = a.indptr[i2 + 1];
        pfY = a.y[i2];
      }
    }
    const PsgdPipeMeta m1 = meta[(q + 1) & 3];
    const int z1 = q + 1 < a.nRows ? m1.z + a.nAug : 0;
    if (tid >= lastWarp0) {
      const int u0 = tid - lastWarp0, u1 = u0 + 32;
      if (u0 < z1) {
        pfJ0 = u0 < m1.z ? a.indices[m1.rb + u0] : (int32_t)(a.d + (u0 - m1.z));
        pfX0 = u0 < m1.z ? a.data[m1.rb + u0] : 1.0;
      }
      if (u1 < z1) {
        pfJ1 = u1 < m1.z ? a.indices[m1.rb + u1] : (int32_t)(a.d + (u1 - m1.z));
        pfX1 = u1 < m1.z ? a.data[m1.rb + u1] : 1.0;
      }
    }
    const long long c0 = clock64();
    // ---- the row's P slice (raw) and the lazy factors of every row feature incl. dummies (psgd.nim:121-127)
    double pv[PSGD_PIPE_R];
    {
      ElemWalk wk = walk0;
#pragma unroll
      for (int r = 0; r < PSGD_PIPE_R; ++r) {
        pv[r] = wk.u < z ? a.P[(int64_t)J[wk.u] * SB8 + wk.off] : 0.0;
        wk.next();
      }
    }
    if (tid < z) {
      const int u = tid;
      const int64_t j = J[u];
      const double sj = a.regScalings[j], tj = a.regThresholds[j];
      sW[u] = u < zReal ? a.w[j] * (scW / a.scalingsW[j]) : 0.0;       // sfm.w[j] *= scaling_w / scalings_w[j]
      sSc[u] = rSc / sj;
      sTh[u] = isL1 ? gamma * rSc * (rTh - tj)                         // l1.nim:89-90
                    : ((rTh - tj) / sj) * gamma;                       // l21.nim:62-63
    }
    // the step sizes (a pow() each: ~1000 dependent FP64 instructions, longer than the load round) are computed ONE
    // SAMPLE AHEAD by three threads of three different warps and parked with the prefetched rows
    double etaNext = 0.0;
    if (tid == nth - 33) etaNext = psgd_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha, it + 1);
    if (tid == nth - 65) etaNext = psgd_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, beta, it + 1);
    if (tid == nth - 97) etaNext = psgd_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha0, it + 1);
    __syncthreads();
    const long long c1 = clock64();
    const double *shEta = sEta + (q & 1) * 4;
    const double etaW = shEta[0], etaP = shEta[1];
    const double etaS = etaP / (1.0 + etaP * beta);                     // psgd.nim:134
    {
      ElemWalk wk = walk0;
#pragma unroll
      for (int r = 0; r < PSGD_PIPE_R; ++r) {
        if (wk.u < z) {
          double p = pv[r];
          if (isL1) {                                                  // l1.nim:86-90
            p *= sSc[wk.u];
            p = psgd_soft(p, sTh[wk.u]);
          }
          sP[tid + r * nth] = p;
        }
        wk.next();
      }
    }
    __syncthreads();
    if (!isL1) {                                                       // l21.nim:60-65: prox, then scale
      if (k <= 32) {
        for (int v = wid; v < z * NO; v += 8 * nw) psgd_l21_prox_warp_x8(sP, v, nw, z * NO, k, NO, sTh, sSc, 0.0);
      } else {
        for (int v = wid; v < z * NO; v += nw) psgd_l21_prox_warp(sP + (size_t)v * k, k, sTh[v / NO], sSc[v / NO]);
      }
      __syncthreads();
    }
    const long long c2 = clock64();
    // ---- predictWithGrad forward (thread <-> (order, component), nonzeros in row order)
    double part = 0.0;
    for (int u = tid; u < zReal; u += nth) part += sW[u] * X[u];
    if (tid < SB8) {
      const int o = tid / k, sc = tid - o * k;
      const int M = a.degree - o;
      AnovaState A;
      part += anova_forward_smem(A, M, sP + o * k + sc, SB8, X, z);
#pragma unroll
      for (int tt = 1; tt < NIMFM_MAX_DEGREE; ++tt)
        if (tt < M) sA[tid * AST + tt] = A[tt];
    }
    const long long c2a = clock64();
    const double yh = block_sum(part, red);
    const long long c2b = clock64();
    if (tid == 0) {
      const double yhat = yh + a.b[0];
      lossAcc += dev_loss(a.cfg.loss, a.cfg.huberThreshold, m.y, yhat);
      sh[4] = dev_dloss(a.cfg.loss, a.cfg.huberThreshold, m.y, yhat);
    }
    __syncthreads();
    const double dL = sh[4];
    const long long c3 = clock64();
    // ---- reg.step (l1.nim:127-136 / l21.nim:102-112), element <-> thread
    {
      ElemWalk wk = walk0;
#pragma unroll 2
      for (int e = tid; e < z * SB8; e += nth) {
        const int u = wk.u, os = wk.off;
        wk.next();
        const int M = sOrd[os];
        const double x = X[u], p = sP[e];
        const double *A = sA + os * AST;
        double g;
        if (M == 2) g = x * (A[1] - p * x);
        else {
          g = x;
          for (int tt = 1; tt < M; tt++) g = x * (A[tt] - p * g);
        }
        const double upd = etaS * (dL * g + beta * p);
        if (isL1) a.P[(int64_t)J[u] * SB8 + os] = psgd_soft(p - upd, gamma * etaS);
        else sP[e] = p - upd;
      }
    }
    if (!isL1) {
      __syncthreads();
      if (k <= 32) {
        for (int v = wid; v < z * NO; v += 8 * nw)
          psgd_l21_prox_warp_x8(sP, v, nw, z * NO, k, NO, nullptr, nullptr, etaS * gamma);
      } else {
        for (int v = wid; v < z * NO; v += nw) psgd_l21_prox_warp(sP + (size_t)v * k, k, etaS * gamma, 1.0);
      }
      __syncthreads();
      ElemWalk wk = walk0;
      for (int e = tid; e < z * SB8; e += nth) {
        a.P[(int64_t)J[wk.u] * SB8 + wk.off] = sP[e];
        wk.next();
      }
    }
    const long long c4 = clock64();
    // ---- reg.updateCacheSGD (l1.nim:106-113 / l21.nim:84-90), w, intercept, caches
    double nSc, nTh;
    if (isL1) {
      nTh = rTh + etaS / rSc;
      nSc = rSc * (1 - etaS * beta);
    } else {
      nTh = rTh + etaP * rSc;
      nSc = rSc / (1 + etaP * beta);
    }
    const double nScW = scW / (1.0 + etaW * alpha);                     // psgd.nim:153
    if (tid < z) {
      const int u = tid;
      const int64_t j = J[u];
      a.regScalings[j] = nSc;
      a.regThresholds[j] = nTh;
      if (u < zReal) {
        if (a.fitLinear) {                                              // fitLinearSGD with eta_w/(1+eta_w*alpha)
          const double eta = etaW / (1.0 + etaW * alpha);
          a.w[j] = sW[u] - eta * (dL * X[u] + alpha * sW[u]);
        }
        a.scalingsW[j] = nScW;
      }
    }
    // ---- park what was fetched ahead
    if (tid == nth - 1) {
      if (q + 3 < a.nRows) meta[(q + 3) & 3].i = pfI;
      if (q + 2 < a.nRows) {
        PsgdPipeMeta &m2 = meta[(q + 2) & 3];
        m2.rb = pfRb;
        m2.z = (int)(pfRe - pfRb);
        m2.y = pfY;
      }
    }
    if (tid >= lastWarp0) {
      int32_t *Jn = sJb + ((q + 1) & 1) * zmax;
      double *Xn = sXb + ((q + 1) & 1) * zmax;
      const int u0 = tid - lastWarp0, u1 = u0 + 32;
      if (u0 < z1) { Jn[u0] = pfJ0; Xn[u0] = pfX0; }
      if (u1 < z1) { Jn[u1] = pfJ1; Xn[u1] = pfX1; }
    }
    if (tid == nth - 33) sEta[((q + 1) & 1) * 4 + 0] = etaNext;
    if (tid == nth - 65) sEta[((q + 1) & 1) * 4 + 1] = etaNext;
    if (tid == nth - 97) sEta[((q + 1) & 1) * 4 + 2] = etaNext;
    if (tid == 0) {                                                     // (sh[1..3] were read before the first barrier)
      if (a.fitIntercept) {                                             // psgd.nim:146-148
        const double e0 = shEta[2];
        const double upd = e0 * (dL + alpha0 * a.b[0]);
        a.b[0] -= upd / (1.0 + e0 * alpha0);
      }
      sh[1] = nSc;
      sh[2] = nTh;
      sh[3] = nScW;
    }
    // ---- resets against underflow (psgd.nim:158-163; l1.nim:116-124 and l21.nim:93-104 as written): rare
    if ((a.fitLinear && nScW < 1e-9) || nSc < 1e-8) {
      __syncthreads();
      if (a.fitLinear && nScW < 1e-9) {
        for (int64_t j = tid; j < a.d; j += nth) {
          double v = a.w[j] * nScW;
          a.w[j] = v / a.scalingsW[j];
          a.scalingsW[j] = 1.0;
        }
        __syncthreads();
        if (tid == 0) sh[3] = 1.0;
        __syncthreads();
      }
      if (nSc < 1e-8) {
        if (isL1) {
          for (int64_t e = tid; e < a.dd * SB8; e += nth) {
            const int64_t j = e / SB8;
            double p = a.P[e] / a.regScalings[j];
            p = psgd_soft(p, gamma * nTh - a.regThresholds[j]);
            a.P[e] = p * nTh;
          }
        } else {
          for (int64_t v = wid; v < a.dd * NO; v += nw) {
            const int64_t j = v / NO;
            const double thr = (nTh - a.regThresholds[j]) / a.regScalings[j];
            psgd_l21_prox_warp(a.P + v * k, k, thr * gamma, nSc / a.regScalings[j]);
          }
        }
        __syncthreads();
        for (int64_t j = tid; j < a.dd; j += nth) {
          a.regScalings[j] = 1.0;
          a.regThresholds[j] = 0.0;
        }
        if (tid == 0) {
          sh[1] = 1.0;
          sh[2] = 0.0;
        }
      }
    }
    __syncthreads();
    if (a.profile && tid == 0) {
      const long long c5 = clock64();
      prof[0] += c1 - c0; prof[1] += c2 - c1; prof[2] += c3 - c2; prof[3] += c4 - c3; prof[4] += c5 - c4;
      prof[5] += c2a - c2; prof[6] += c2b - c2a;
    }
  }
  if (a.profile && tid == 0 && a.nRows > 0)
    printf("psgd pipe cycles/sample: loads %lld  lazy %lld  forward %lld (dp %lld, sum %lld)  step %lld  caches+park %lld\n",
           prof[0] / a.nRows, prof[1] / a.nRows, prof[2] / a.nRows, prof[5] / a.nRows, prof[6] / a.nRows,
           prof[3] / a.nRows, prof[4] / a.nRows);
  lossAcc = block_sum(lossAcc, red);
  if (tid == 0) {
    a.scal[0] = sh[1];
    a.scal[1] = sh[2];
    a.scal[2] = sh[3];
    a.scal[3] = lossAcc;
  }
}

// finalize (psgd.nim:58-75): w catch-up, reg.lazyUpdateFinal (l1.nim:93-103 resets its caches,
// l21.nim:68-75 does not)
__global__ void __launch_bounds__(PSGD_THREADS, 1) psgd_finalize_kernel(const PsgdArgs a) {
  const int k = a.k, NO = a.nOrders, SB8 = NO * k;
  const int tid = threadIdx.x, nth = blockDim.x, wid = tid >> 5, nw = nth >> 5;
  const double rSc = a.scal[0], rTh = a.scal[1], scW = a.scal[2], gamma = a.cfg.gamma;
  __syncthreads();
  if (a.fitLinear)
    for (int64_t j = tid; j < a.d; j += nth) {
      double v = a.w[j] * scW;
      a.w[j] = v / a.scalingsW[j];
      a.scalingsW[j] = scW;
    }
  if (a.cfg.reg == NIMFM_REG_L1) {
    for (int64_t e = tid; e < a.dd * SB8; e += nth) {
      const int64_t j = e / SB8;
      double p = a.P[e] * (rSc / a.regScalings[j]);
      a.P[e] = psgd_soft(p, gamma * rSc * (rTh - a.regThresholds[j]));
    }
    __syncthreads();
    for (int64_t j = tid; j < a.dd; j += nth) {
      a.regScalings[j] = 1.0;
      a.regThresholds[j] = 0.0;
    }
    if (tid == 0) {
      a.scal[0] = 1.0;
      a.scal[1] = 0.0;
    }
  } else if (a.cfg.reg == NIMFM_REG_L21) {
    for (int64_t v = wid; v < a.dd * NO; v += nw) {
      const int64_t j = v / NO;
      const double thr = (rTh - a.regThresholds[j]) / a.regScalings[j];
      psgd_l21_prox_warp(a.P + v * k, k, thr * gamma, rSc / a.regScalings[j]);
    }
  }
}

// dense step of the SquaredL12 route (squaredl12.nim:224-228 for P; the eager equivalent of the lazily
// scaled w of psgd.nim:122-155; the intercept of :146-148).  g = dL*dA scattered by the row kernel; tail = [dL, loss]
static __global__ void psgd_dense_step_kernel(double *P, double *gP, int64_t nP, double etaS, double beta, double *w,
                                              double *gw, int64_t d, double etaW, double alpha, int fitLinear,
                                              double *b, double *tail, double eta0v, double alpha0,
                                              int fitIntercept, double *lossAcc) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t tid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  for (int64_t e = tid; e < nP; e += stride) {
    const double p = P[e];
    P[e] = p - etaS * (gP[e] + beta * p);
    gP[e] = 0.0;
  }
  const double etaWs = etaW / (1.0 + etaW * alpha), rW = 1.0 / (1.0 + etaW * alpha);
  for (int64_t j = tid; j < d; j += stride) {
    if (fitLinear) {
      const double g = gw[j], wv = w[j];
      // touched: w - eta'(dL x + alpha w); untouched: only the lazy scaling 1/(1+eta_w alpha) (== 1 - eta' alpha)
      w[j] = g != 0.0 ? wv - etaWs * (g + alpha * wv) : wv * rW;
    }
    gw[j] = 0.0;
  }
  if (tid == 0) {
    if (fitIntercept) {
      const double upd = eta0v * (tail[0] + alpha0 * b[0]);
      b[0] -= upd / (1.0 + eta0v * alpha0);
    }
    lossAcc[0] += tail[1];
    tail[0] = 0.0;
    tail[1] = 0.0;
  }
}

static void psgd_fill(nimfm_ctx *ctx, double *p, int64_t n, double v) {
  fill_kernel<<<ew_grid(ctx, n), 256, 0, ctx->stream>>>(p, n, v);
  LAUNCHED(ctx);
}

extern "C" {

// reg.initSGD + the scaling caches of PSGD.fit (psgd.nim:98-112)
int32_t nimfm_fm_psgd_begin(nimfm_ctx *ctx, nimfm_fm *fm) {
  if (!ctx || !fm) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  const int64_t dd = fm->dd(), d = fm->d;
  if (!fm->scalingsP) {
    CK(cudaMalloc(&fm->scalingsP, (size_t)dd * 8));
    CK(cudaMalloc(&fm->scalingsW, (size_t)d * 8));
    CK(cudaMalloc(&fm->sgdScal, 8 * 8));
  }
  if (!fm->psgdThr) CK(cudaMalloc(&fm->psgdThr, (size_t)dd * 8));
  psgd_fill(ctx, fm->scalingsP, dd, 1.0);
  psgd_fill(ctx, fm->scalingsW, d, 1.0);
  psgd_fill(ctx, fm->psgdThr, dd, 0.0);
  const double sc[4] = {1.0, 0.0, 1.0, 0.0};   // reg scaling, reg threshold, scaling_w, loss
  CK(cudaMemcpyAsync(fm->sgdScal, sc, 32, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(fm->grad, 0, (size_t)(fm->nP() + d + 2) * 8, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  fm->psgdReady = true;
  return NIMFM_OK;
}

int32_t nimfm_fm_psgd_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_psgd_cfg *cfg,
                            int64_t *it, const int64_t *perm, int64_t nRows, double *lossSum) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(fm && X && cfg && it, "NULL argument");
  if (!fm->psgdReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_fm_psgd_begin was not called");
  REQUIRE(X->kind != NIMFM_DS_CSC, "a CSR dataset is required");
  REQUIRE(X->d == fm->d, "Invalid nFeatures.");
  REQUIRE(X->y != nullptr, "dataset has no targets");
  REQUIRE(nRows >= 0 && (perm || nRows <= X->n), "bad nRows");
  REQUIRE(cfg->reg >= NIMFM_REG_L1 && cfg->reg <= NIMFM_REG_L21, "unsupported regulariser");
  const bool sq = cfg->reg == NIMFM_REG_SQUAREDL12 || cfg->reg == NIMFM_REG_SQUAREDL12_ROWS;
  REQUIRE(!(sq && fm->degree != 2), "SquaredL12 supports only degree=2.");      // squaredl12.nim:103-106
  CK(cudaSetDevice(ctx->device));
  int rc;
  const int64_t nP = fm->nP(), d = fm->d, nG = nP + d + 2;
  CK(cudaMemsetAsync(fm->sgdScal + 3, 0, 8, ctx->stream));
  if (!sq) {
    const int32_t *permDev = nullptr;
    if (perm && nRows > 0) {
      if ((rc = nimfm_stage_row_ids(ctx, perm, nRows, X->n))) return rc;
      permDev = ctx->idx32Scratch;
    }
    const int SB8 = fm->nOrders * fm->k;
    const int zmax = (int)std::max<int64_t>(X->maxSegNnz + fm->nAug, 1);
    const size_t smem = ((size_t)zmax * SB8 + 4 * (size_t)zmax) * 8 + (size_t)zmax * 8;
    if (SB8 > PSGD_THREADS || smem > (size_t)ctx->smemOptin - 2048)
      return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED,
                        "PSGD: nOrders*nComponents=%d (max %d) or a %d-nonzero row's slice (%zu B) does not fit", SB8,
                        PSGD_THREADS, zmax, smem);
    PsgdArgs a;
    memset(&a, 0, sizeof(a));
    a.data = X->data; a.indices = X->indices; a.indptr = X->indptr; a.y = X->y; a.perm = permDev;
    a.nRows = nRows; a.d = d; a.dd = fm->dd();
    a.degree = fm->degree; a.k = fm->k; a.nOrders = fm->nOrders; a.nAug = fm->nAug;
    a.fitLinear = fm->fitLinear; a.fitIntercept = fm->fitIntercept;
    a.P = fm->P; a.w = fm->w; a.b = fm->b;
    a.regScalings = fm->scalingsP; a.regThresholds = fm->psgdThr; a.scalingsW = fm->scalingsW; a.scal = fm->sgdScal;
    a.cfg = *cfg; a.it0 = *it; a.zmax = zmax;
    const size_t smemPipe = ((size_t)zmax * SB8 + (size_t)SB8 * (NIMFM_MAX_DEGREE + 1) + 5 * (size_t)zmax) * 8 +
                            2 * (size_t)zmax * 4 + (size_t)SB8 + 16;
    const char *env = getenv("NIMFM_PSGD_KERNEL");   // "staged": the unpipelined kernel
    // degree 1 (SB8 = 0, no P) takes the staged kernel, whose P passes are empty loops; the pipelined one divides by SB8
    if (SB8 > 0 && zmax <= 64 && (size_t)zmax * SB8 <= (size_t)PSGD_PIPE_R * PSGD_PIPE_THREADS &&
        smemPipe + 4096 <= (size_t)ctx->smemOptin && !(env && env[0] == 's')) {
      a.profile = getenv("NIMFM_PSGD_PROFILE") != nullptr;
      CK(cudaFuncSetAttribute(psgd_lazy_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemPipe));
      psgd_lazy_pipe_kernel<<<1, PSGD_PIPE_THREADS, smemPipe, ctx->stream>>>(a);
    } else {
      CK(cudaFuncSetAttribute(psgd_lazy_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      psgd_lazy_kernel<<<1, PSGD_THREADS, smem, ctx->stream>>>(a);
    }
    LAUNCHED(ctx);
  } else {
    for (int64_t q = 0; q < nRows; q++) {
      const int64_t i = perm ? perm[q] : q;
      REQUIRE(i >= 0 && i < X->n, "row id %lld out of range", (long long)i);
      const int64_t itq = *it + q;
      if ((rc = nimfm_fm_loss_grad_one_row(ctx, fm, X, cfg->loss, cfg->huberThreshold, i))) return rc;
      const double etaW = host_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha, itq);
      const double etaP = host_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->beta, itq);
      const double eta0v = host_eta(cfg->scheduling, cfg->eta0, cfg->power, cfg->alpha0, itq);
      const double etaS = etaP / (1.0 + etaP * cfg->beta);
      psgd_dense_step_kernel<<<ew_grid(ctx, nP), 256, 0, ctx->stream>>>(
          fm->P, fm->grad, nP, etaS, cfg->beta, fm->w, fm->grad + nP, d, etaW, cfg->alpha, fm->fitLinear, fm->b,
          fm->grad + nG - 2, eta0v, cfg->alpha0, fm->fitIntercept, fm->sgdScal + 3);
      LAUNCHED(ctx);
      if ((rc = nimfm_fm_apply_prox(ctx, fm, cfg->reg, cfg->gamma * etaS))) return rc;
    }
  }
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ctx->hostScalars, fm->sgdScal, 32, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *it += nRows;
  if (lossSum) *lossSum = ctx->hostScalars[3];
  return NIMFM_OK;
}

// finalize(self, sfm, P, scaling_w, scalings_w) (psgd.nim:58-75); a no-op for the eager SquaredL12 route
int32_t nimfm_fm_psgd_end(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_psgd_cfg *cfg) {
  if (!ctx || !fm || !cfg) return NIMFM_ERR_INVALID;
  if (!fm->psgdReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_fm_psgd_begin was not called");
  CK(cudaSetDevice(ctx->device));
  if (cfg->reg == NIMFM_REG_L1 || cfg->reg == NIMFM_REG_L21) {
    PsgdArgs a;
    memset(&a, 0, sizeof(a));
    a.d = fm->d; a.dd = fm->dd(); a.k = fm->k; a.nOrders = fm->nOrders; a.fitLinear = fm->fitLinear;
    a.P = fm->P; a.w = fm->w;
    a.regScalings = fm->scalingsP; a.regThresholds = fm->psgdThr; a.scalingsW = fm->scalingsW; a.scal = fm->sgdScal;
    a.cfg = *cfg;
    psgd_finalize_kernel<<<1, PSGD_THREADS, 0, ctx->stream>>>(a);
    LAUNCHED(ctx);
  }
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  return NIMFM_OK;
}

}  // extern "C"
