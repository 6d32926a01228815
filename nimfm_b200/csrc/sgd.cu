// sgd.cu -- SGD with lazy L2 scaling for FM (optimizer/sgd.nim:99-143, 205-258) and FFM
// (optimizer/sgd_ffm.nim:11-46), SURVEY K6.
//
// SGD is strictly sequential per sample: step i reads the parameters step i-1 wrote (through P, w,
// the intercept and the global scaling_P / scaling_w).  The device therefore runs the whole sample
// loop inside ONE persistent thread block (the parallelism is inside a row: threads <-> (order,
// component) for FM, (nonzero, component) for FFM) and keeps the reference's exact semantics.
// "Replicas only" for multi-GPU; the data-parallel solvers are MBPSGD and minibatch AdaGrad.
#include <math.h>
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"

#define SGD_THREADS 256

__device__ __forceinline__ double dev_eta(int sched, double eta0, double power, double reg, int64_t it) {
  switch (sched) {  // getEta, sgd.nim:60-69
    case NIMFM_SCHED_CONSTANT: return eta0;
    case NIMFM_SCHED_OPTIMAL: return eta0 / pow(1.0 + eta0 * reg * (double)it, power);
    case NIMFM_SCHED_INVSCALING: return eta0 / pow((double)it, power);
    default: return 1.0 / (reg * (double)it);
  }
}

struct SgdArgs {
  const double *data;
  const int32_t *indices, *fields;
  const int64_t *indptr;
  const double *y;
  const int32_t *perm;
  int64_t nRows, d, dd;
  int degree, k, nOrders, nAug, nFields;
  int fitLinear, fitIntercept;
  double *P, *w, *b;
  double *scalingsP, *scalingsW, *scal;   // scal: [scaling_P, scaling_w, viol, loss]
  double *dA;                             // FFM scratch: [zmax][nFields][k]
  nimfm_sgd_cfg cfg;
  int64_t it0;
};

// dense pass of finalize / resetScaling (sgd.nim:99-131).  SB8 = doubles per feature slice.
__device__ void sgd_materialize(const SgdArgs &a, int SB8, int64_t nFeatP, bool doW, bool doP, double scP,
                                double scW) {
  if (doW && a.fitLinear)
    for (int64_t j = threadIdx.x; j < a.d; j += blockDim.x) {
      double v = a.w[j] * scW;
      a.w[j] = v / a.scalingsW[j];
      a.scalingsW[j] = 1.0;
    }
  if (doP) {
    for (int64_t e = threadIdx.x; e < nFeatP * SB8; e += blockDim.x) {
      const int64_t j = e / SB8;
      a.P[e] *= scP / a.scalingsP[j];
    }
    __syncthreads();
    for (int64_t j = threadIdx.x; j < a.dd; j += blockDim.x) a.scalingsP[j] = 1.0;
  }
  __syncthreads();
}

template <bool FFM>
__global__ void __launch_bounds__(SGD_THREADS, 1) sgd_epoch_kernel(const SgdArgs a) {
  __shared__ double red[SGD_THREADS / 32];
  __shared__ double sh[4];   // yhat, scaling_P, scaling_w, dL
  const int k = a.k;
  const int NO = FFM ? a.nFields : a.nOrders;
  const int SB8 = NO * k;
  const int tid = threadIdx.x, nth = blockDim.x;
  double viol = 0.0, lossAcc = 0.0;
  if (tid == 0) {
    sh[1] = a.scal[0];
    sh[2] = a.scal[1];
  }
  __syncthreads();
  const double alpha0 = a.cfg.alpha0, alpha = a.cfg.alpha, beta = a.cfg.beta;
  for (int64_t q = 0; q < a.nRows; ++q) {
    const int64_t i = a.perm ? (int64_t)a.perm[q] : q;
    const int64_t it = a.it0 + q;
    const int64_t rb = a.indptr[i];
    const int zReal = (int)(a.indptr[i + 1] - rb);
    const int z = zReal + (FFM ? 0 : a.nAug);
    const double scP = sh[1], scW = sh[2];
    // ---- lazilyUpdate (sgd.nim:134-143): real features only
    for (int e = tid; e < zReal * SB8; e += nth) {
      const int u = e / SB8, off = e - u * SB8;
      const int64_t j = a.indices[rb + u];
      a.P[j * SB8 + off] *= scP / a.scalingsP[j];
    }
    if (a.fitLinear)
      for (int u = tid; u < zReal; u += nth) {
        const int64_t j = a.indices[rb + u];
        a.w[j] *= scW / a.scalingsW[j];
      }
    __syncthreads();
    // ---- predictWithGrad: forward
    double part = 0.0;
    for (int u = tid; u < zReal; u += nth) part += a.w[a.indices[rb + u]] * a.data[rb + u];
    if (!FFM) {
      for (int os = tid; os < SB8; os += nth) {          // thread <-> (order, component)
        const int o = os / k, s = os - o * k;
        const int M = a.degree - o;
        AnovaState A;
        anova_init(A);
        for (int u = 0; u < z; u++) {
          const int64_t j = u < zReal ? (int64_t)a.indices[rb + u] : a.d + (u - zReal);
          const double x = u < zReal ? a.data[rb + u] : 1.0;
          const double tv = a.P[j * SB8 + o * k + s] * x;
          if (M == 2) {
            A[1] += tv;
            A[2] += tv * tv;
          } else {
            anova_step(A, M, tv);
          }
        }
        if (M == 2) A[2] = (A[1] * A[1] - A[2]) / 2.0;
        part += anova_at(A, M);
      }
    } else {
      // dA[u][f][s] = sum_{b != u, field_b == f} x_u x_b P[j_b][f_u][s]   (sgd_ffm.nim:18-30)
      for (int e = tid; e < zReal * SB8; e += nth) a.dA[e] = 0.0;
      __syncthreads();
      for (int us = tid; us < zReal * k; us += nth) {    // thread <-> (nonzero, component)
        const int u = us / k, s = us - u * k;
        const int fu = a.fields[rb + u];
        const double xu = a.data[rb + u];
        for (int v = 0; v < zReal; v++) {
          if (v == u) continue;
          const int64_t jv = a.indices[rb + v];
          const int fv = a.fields[rb + v];
          a.dA[((size_t)u * NO + fv) * k + s] += (xu * a.data[rb + v]) * a.P[jv * SB8 + fu * k + s];
        }
      }
      __syncthreads();
      double pp = 0.0;
      for (int e = tid; e < zReal * SB8; e += nth) {
        const int u = e / SB8, off = e - u * SB8;
        pp += a.P[(int64_t)a.indices[rb + u] * SB8 + off] * a.dA[e];
      }
      part += 0.5 * pp;
    }
    double yhat = block_sum(part, red);
    if (tid == 0) {
      yhat += a.b[0];
      sh[0] = yhat;
      const double yi = a.y[i];
      lossAcc += dev_loss(a.cfg.loss, a.cfg.huberThreshold, yi, yhat);
      sh[3] = dev_dloss(a.cfg.loss, a.cfg.huberThreshold, yi, yhat);
    }
    __syncthreads();
    const double dL = sh[3];
    // ---- update (sgd.nim:205-243)
    const double etaW = dev_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha, it);
    const double etaP = dev_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, beta, it);
    if (!FFM) {
      for (int os = tid; os < SB8; os += nth) {
        const int o = os / k, s = os - o * k;
        const int M = a.degree - o;
        // recompute the DP state of this (order, component), then the derivative recurrence (sgd.nim:176-188)
        AnovaState A;
        anova_init(A);
        for (int u = 0; u < z; u++) {
          const int64_t j = u < zReal ? (int64_t)a.indices[rb + u] : a.d + (u - zReal);
          const double x = u < zReal ? a.data[rb + u] : 1.0;
          const double tv = a.P[j * SB8 + o * k + s] * x;
          if (M == 2) A[1] += tv;
          else
            anova_step(A, M, tv);
        }
        for (int u = 0; u < z; u++) {
          const int64_t j = u < zReal ? (int64_t)a.indices[rb + u] : a.d + (u - zReal);
          const double x = u < zReal ? a.data[rb + u] : 1.0;
          const int64_t e = j * SB8 + o * k + s;
          const double p = a.P[e];
          double g;
          if (M == 2) g = x * (A[1] - p * x);
          else {
            g = anova_deriv(A, M, x, p);
          }
          const double upd = etaP * (dL * g + beta * p);
          viol += fabs(upd);
          a.P[e] = p - upd;
        }
      }
    } else {
      for (int e = tid; e < zReal * SB8; e += nth) {
        const int u = e / SB8, off = e - u * SB8;
        const int64_t pe = (int64_t)a.indices[rb + u] * SB8 + off;
        const double p = a.P[pe];
        const double upd = etaP * (dL * a.dA[e] + beta * p);
        viol += fabs(upd);
        a.P[pe] = p - upd;
      }
    }
    if (a.fitLinear)                                        // fitLinearSGD, fit_linear.nim:41-47
      for (int u = tid; u < zReal; u += nth) {
        const int64_t j = a.indices[rb + u];
        const double upd = etaW * (dL * a.data[rb + u] + alpha * a.w[j]);
        a.w[j] -= upd;
        viol += fabs(upd);
      }
    const double nscP = scP * (1 - etaP * beta), nscW = scW * (1 - etaW * alpha);
    for (int u = tid; u < zReal; u += nth) {
      const int64_t j = a.indices[rb + u];
      a.scalingsP[j] = nscP;
      a.scalingsW[j] = nscW;
    }
    if (!FFM)
      for (int u = tid; u < a.nAug; u += nth) a.scalingsP[a.d + u] = nscP;
    if (tid == 0) {
      if (a.fitIntercept) {
        const double upd = dev_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha0, it) * (dL + alpha0 * a.b[0]);
        viol += fabs(upd);
        a.b[0] -= upd;
      }
      sh[1] = nscP;
      sh[2] = nscW;
    }
    __syncthreads();
    // ---- resetScaling (sgd.nim:116-131)
    const bool resetW = a.fitLinear && nscW < 1e-9, resetP = nscP < 1e-9;
    if (resetW || resetP) {
      sgd_materialize(a, SB8, a.d, resetW, resetP, nscP, nscW);   // P: features 0..d-1 only (:126)
      if (tid == 0) {
        if (resetW) sh[2] = 1.0;
        if (resetP) sh[1] = 1.0;
      }
      __syncthreads();
    }
  }
  viol = block_sum(viol, red);
  __syncthreads();
  lossAcc = block_sum(lossAcc, red);
  if (tid == 0) {
    a.scal[0] = sh[1];
    a.scal[1] = sh[2];
    a.scal[2] = viol;
    a.scal[3] = lossAcc;
  }
}

// FM sample loop with the row's P slice STAGED IN SHARED MEMORY: the unstaged loop above walks a row's
// nonzeros with one dependent global load per step of the DP (39 L2 round trips per pass, 36 us per
// C4 sample); here the z*nOrders*k doubles are fetched by all threads at once (lazy scaling applied on
// the way in), the DP and the derivative recurrence run out of shared memory, and the updated slice
// is written back coalesced.  Same operations in the same order per element as sgd_epoch_kernel<false>.
// dynamic smem: sP[zmax*SB8] | sX[zmax] | sW[zmax] | sSc[zmax] | sJ[zmax] (int64)
__global__ void __launch_bounds__(SGD_THREADS, 1) sgd_fm_staged_kernel(const SgdArgs a, int zmax) {
  extern __shared__ __align__(16) unsigned char sgd_smem[];
  __shared__ double red[SGD_THREADS / 32];
  __shared__ double sh[4];   // yhat, scaling_P, scaling_w, dL
  const int k = a.k, NO = a.nOrders, SB8 = NO * k;
  double *sP = reinterpret_cast<double *>(sgd_smem);
  double *sX = sP + (size_t)zmax * SB8;
  double *sW = sX + zmax;
  double *sSc = sW + zmax;
  int64_t *sJ = reinterpret_cast<int64_t *>(sSc + zmax);
  const int tid = threadIdx.x, nth = blockDim.x;
  double viol = 0.0, lossAcc = 0.0;
  if (tid == 0) {
    sh[1] = a.scal[0];
    sh[2] = a.scal[1];
  }
  __syncthreads();
  const double alpha0 = a.cfg.alpha0, alpha = a.cfg.alpha, beta = a.cfg.beta;
  for (int64_t q = 0; q < a.nRows; ++q) {
    const int64_t i = a.perm ? (int64_t)a.perm[q] : q;
    const int64_t it = a.it0 + q;
    const int64_t rb = a.indptr[i];
    const int zReal = (int)(a.indptr[i + 1] - rb);
    const int z = zReal + a.nAug;
    const double scP = sh[1], scW = sh[2];
    // ---- records; lazilyUpdate factors (sgd.nim:134-143: real features only)
    for (int u = tid; u < z; u += nth) {
      if (u < zReal) {
        const int64_t j = a.indices[rb + u];
        sJ[u] = j;
        sX[u] = a.data[rb + u];
        sSc[u] = scP / a.scalingsP[j];
        double wv = a.w[j];
        if (a.fitLinear) wv *= scW / a.scalingsW[j];
        sW[u] = wv;
      } else {
        sJ[u] = a.d + (u - zReal);
        sX[u] = 1.0;
        sSc[u] = 1.0;
        sW[u] = 0.0;
      }
    }
    __syncthreads();
    for (int e = tid; e < z * SB8; e += nth) {
      const int u = e / SB8, off = e - u * SB8;
      double p = a.P[sJ[u] * SB8 + off];
      if (u < zReal) p *= sSc[u];
      sP[e] = p;
    }
    __syncthreads();
    // ---- predictWithGrad: forward (thread <-> (order, component)); A stays in registers for the update
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
      sh[3] = dev_dloss(a.cfg.loss, a.cfg.huberThreshold, yi, yhat);
    }
    __syncthreads();
    const double dL = sh[3];
    // ---- update (sgd.nim:205-243)
    const double etaW = dev_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha, it);
    const double etaP = dev_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, beta, it);
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
        const double upd = etaP * (dL * g + beta * p);
        viol += fabs(upd);
        sP[e] = p - upd;
      }
    }
    const double nscP = scP * (1 - etaP * beta), nscW = scW * (1 - etaW * alpha);
    for (int u = tid; u < zReal; u += nth) {
      const int64_t j = sJ[u];
      if (a.fitLinear) {                                    // fitLinearSGD, fit_linear.nim:41-47
        const double upd = etaW * (dL * sX[u] + alpha * sW[u]);
        a.w[j] = sW[u] - upd;
        viol += fabs(upd);
      }
      a.scalingsP[j] = nscP;
      a.scalingsW[j] = nscW;
    }
    for (int u = tid; u < a.nAug; u += nth) a.scalingsP[a.d + u] = nscP;
    __syncthreads();
    for (int e = tid; e < z * SB8; e += nth) {
      const int u = e / SB8, off = e - u * SB8;
      a.P[sJ[u] * SB8 + off] = sP[e];
    }
    if (tid == 0) {
      if (a.fitIntercept) {
        const double upd = dev_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha0, it) * (dL + alpha0 * a.b[0]);
        viol += fabs(upd);
        a.b[0] -= upd;
      }
      sh[1] = nscP;
      sh[2] = nscW;
    }
    __syncthreads();
    // ---- resetScaling (sgd.nim:116-131)
    const bool resetW = a.fitLinear && nscW < 1e-9, resetP = nscP < 1e-9;
    if (resetW || resetP) {
      sgd_materialize(a, SB8, a.d, resetW, resetP, nscP, nscW);
      if (tid == 0) {
        if (resetW) sh[2] = 1.0;
        if (resetP) sh[1] = 1.0;
      }
      __syncthreads();
    }
  }
  viol = block_sum(viol, red);
  __syncthreads();
  lossAcc = block_sum(lossAcc, red);
  if (tid == 0) {
    a.scal[0] = sh[1];
    a.scal[1] = sh[2];
    a.scal[2] = viol;
    a.scal[3] = lossAcc;
  }
}

// The FM sample loop, PIPELINED (the default): the staged kernel above spends most of a sample waiting on a chain of
// dependent global loads (permutation -> indptr -> indices / values -> scalings, w -> P rows: 23 us per C4 sample,
// 43 K samples/s -- slower than one host core on the same loop).  Here
//   * the CSR side of the chain is read-only, so it is fetched AHEAD: the last warp loads sample q+2's row pointer
//     and target and sample q+1's indices / values into a second set of shared buffers while sample q computes;
//   * what depends on the previous update (scalings, w, the P rows) is one round of independent loads issued by all
//     512 threads at once; eta (a pow()) is computed by one otherwise idle thread in that shadow;
//   * the forward DP keeps the reference's order (thread <-> (order, component), nonzeros in row order), leaves
//     A[.][1..M-1] in shared memory, and the derivative + update + write-back is spread over ALL threads
//     (element <-> thread), straight from shared memory to global.
// Same arithmetic per parameter element as sgd_epoch_kernel<false>; viol is summed in a different order.
// dynamic smem: sP[zmax*SB8] | sA[SB8*(MAXDEG+1)] | sX[2][zmax] | sW[zmax] | sSc[zmax] | sJ[2][zmax] (int32) | sOrd[SB8]
#define SGDP_THREADS 512
#define SGDP_R 12                       // row slice elements per thread: zmax * SB8 <= SGDP_R * SGDP_THREADS
struct SgdPipeMeta {
  int64_t i, rb;
  double y;
  int z;
};

__global__ void __launch_bounds__(SGDP_THREADS, 1) sgd_fm_pipe_kernel(const SgdArgs a, int zmax) {
  extern __shared__ __align__(16) unsigned char sgd_smem[];
  __shared__ double red[SGDP_THREADS / 32];
  __shared__ double sh[8];              // [1] scaling_P, [2] scaling_w, [3] dL
  __shared__ SgdPipeMeta meta[4];       // ring: sample q lives in meta[q & 3]
  __shared__ double sEta[8];            // [q & 1][eta_P, eta_w, eta_b, -]
  const int k = a.k, NO = a.nOrders, SB8 = NO * k, AST = NIMFM_MAX_DEGREE + 1;
  double *sP = reinterpret_cast<double *>(sgd_smem);
  double *sA = sP + (size_t)zmax * SB8;
  double *sXb = sA + (size_t)SB8 * AST;
  double *sW = sXb + 2 * (size_t)zmax;
  double *sSc = sW + zmax;
  int32_t *sJb = reinterpret_cast<int32_t *>(sSc + zmax);
  const int tid = threadIdx.x, nth = blockDim.x;
  const int lastWarp0 = nth - 32;       // the prefetching warp
  double viol = 0.0, lossAcc = 0.0;
  long long prof[4] = {0, 0, 0, 0};
  const double alpha0 = a.cfg.alpha0, alpha = a.cfg.alpha, beta = a.cfg.beta;
  ElemWalk walk0;                       // (u, off) of this thread's elements of a row slice without divisions
  walk0.start(tid, nth, SB8);
  signed char *sOrd = reinterpret_cast<signed char *>(sJb + 2 * zmax);   // [SB8] ANOVA order of (order, component) slot
  for (int os = tid; os < SB8; os += nth) sOrd[os] = (signed char)(a.degree - os / k);

  // prologue: the read-only chain of the first samples, loaded the plain way
  if (tid == 32) {
    sEta[0] = dev_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, beta, a.it0);
    sEta[1] = dev_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha, a.it0);
    sEta[2] = dev_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha0, a.it0);
  }
  if (tid == 0) {
    sh[1] = a.scal[0];
    sh[2] = a.scal[1];
    for (int64_t q = 0; q < 3 && q < a.nRows; ++q) {
      SgdPipeMeta m;
      m.i = a.perm ? (int64_t)a.perm[q] : q;
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
    const SgdPipeMeta m = meta[0];
    for (int u = tid - lastWarp0; u < m.z + a.nAug; u += 32) {
      sJb[u] = u < m.z ? a.indices[m.rb + u] : (int32_t)(a.d + (u - m.z));
      sXb[u] = u < m.z ? a.data[m.rb + u] : 1.0;
    }
  }
  __syncthreads();

  for (int64_t q = 0; q < a.nRows; ++q) {
    const int64_t it = a.it0 + q;
    const SgdPipeMeta m = meta[q & 3];
    const int zReal = m.z, z = zReal + a.nAug;
    // ---- the read-only side of the chain, fetched AHEAD into registers by the last warp; each stage is a single
    // level of loads issued here and parked in shared memory at the END of the iteration, so the warp never waits
    // on them before the block's barriers: sample q+3's row id, q+2's row pointer / target, q+1's indices / values
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
    const SgdPipeMeta m1 = meta[(q + 1) & 3];
    const int z1 = q + 1 < a.nRows ? m1.z + a.nAug : 0;
    if (tid >= lastWarp0) {                                  // up to 64 nonzeros per row through this path
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
    const int32_t *J = sJb + (q & 1) * zmax;
    const double *X = sXb + (q & 1) * zmax;
    const double scP = sh[1], scW = sh[2];
    long long c0 = clock64();
    // ---- phase 1: everything that depends on the previous update, in one round of independent loads
    if (tid < z) {
      if (tid < zReal) {
        const int64_t j = J[tid];
        sSc[tid] = scP / a.scalingsP[j];                    // lazilyUpdate, sgd.nim:134-143 (real features only)
        double wv = a.w[j];
        if (a.fitLinear) wv *= scW / a.scalingsW[j];
        sW[tid] = wv;
      } else {
        sSc[tid] = 1.0;
        sW[tid] = 0.0;
      }
    }
    double pr[SGDP_R];                                       // the row's P slice: all loads before the first use (one
    {                                                        // memory latency, not one per element), held in registers
      ElemWalk wk = walk0;                                   // until the lazy factors are in shared memory
#pragma unroll
      for (int r = 0; r < SGDP_R; ++r) {
        pr[r] = wk.u < z ? a.P[(int64_t)J[wk.u] * SB8 + wk.off] : 0.0;
        wk.next();
      }
    }
    // the step sizes (a pow() each: ~1000 dependent FP64 instructions, longer than the load round above) are computed
    // ONE SAMPLE AHEAD by three threads of three different warps and parked with the prefetched rows
    double etaNext = 0.0;
    if (tid == nth - 33) etaNext = dev_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, beta, it + 1);
    if (tid == nth - 65) etaNext = dev_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha, it + 1);
    if (tid == nth - 97) etaNext = dev_eta(a.cfg.scheduling, a.cfg.eta0, a.cfg.power, alpha0, it + 1);
    __syncthreads();
    long long c1 = clock64();
    {
      ElemWalk wk = walk0;
#pragma unroll
      for (int r = 0; r < SGDP_R; ++r) {
        if (wk.u < z) sP[tid + r * nth] = wk.u < zReal ? pr[r] * sSc[wk.u] : pr[r];
        wk.next();
      }
    }
    __syncthreads();
    // ---- predictWithGrad: forward, thread <-> (order, component), nonzeros in row order (sgd.nim:146-173)
    double part = 0.0;
    for (int u = tid; u < zReal; u += nth) part += sW[u] * X[u];
    if (tid < SB8) {
      const int o = tid / k, sc = tid - o * k;
      const int M = a.degree - o;
      AnovaState A;
      part += anova_forward_smem(A, M, sP + o * k + sc, SB8, X, z);
#pragma unroll
      for (int t = 1; t < NIMFM_MAX_DEGREE; ++t)
        if (t < M) sA[tid * AST + t] = A[t];
    }
    long long c2 = clock64();
    const double yh = block_sum(part, red);
    if (tid == 0) {
      const double yhat = yh + a.b[0];
      lossAcc += dev_loss(a.cfg.loss, a.cfg.huberThreshold, m.y, yhat);
      sh[3] = dev_dloss(a.cfg.loss, a.cfg.huberThreshold, m.y, yhat);
    }
    __syncthreads();
    const double *shEta = sEta + (q & 1) * 4;
    const double dL = sh[3], etaP = shEta[0], etaW = shEta[1];
    long long c3 = clock64();
    // ---- update (sgd.nim:205-243): element <-> thread, derivative recurrence from the stored A (sgd.nim:176-188)
    ElemWalk wu = walk0;
#pragma unroll 2
    for (int e = tid; e < z * SB8; e += nth) {
      const int u = wu.u, os = wu.off;
      wu.next();
      const int M = sOrd[os];
      const double x = X[u], p = sP[e];
      const double *A = sA + os * AST;
      double g;
      if (M == 2) g = x * (A[1] - p * x);
      else {
        g = x;
        for (int t = 1; t < M; t++) g = x * (A[t] - p * g);   // A in shared memory: dynamic indexing is fine here
      }
      const double upd = etaP * (dL * g + beta * p);
      viol += fabs(upd);
      a.P[(int64_t)J[u] * SB8 + os] = p - upd;
    }
    const double nscP = scP * (1 - etaP * beta), nscW = scW * (1 - etaW * alpha);
    if (tid < zReal) {
      const int64_t j = J[tid];
      if (a.fitLinear) {                                    // fitLinearSGD, fit_linear.nim:41-47
        const double upd = etaW * (dL * X[tid] + alpha * sW[tid]);
        a.w[j] = sW[tid] - upd;
        viol += fabs(upd);
      }
      a.scalingsP[j] = nscP;
      a.scalingsW[j] = nscW;
    } else if (tid < z) {
      a.scalingsP[a.d + (tid - zReal)] = nscP;
    }
    if (tid == 0) {
      if (a.fitIntercept) {
        const double upd = shEta[2] * (dL + alpha0 * a.b[0]);
        viol += fabs(upd);
        a.b[0] -= upd;
      }
      sh[1] = nscP;
      sh[2] = nscW;
    }
    // ---- park what was fetched ahead (the slots being written belong to samples q+1 .. q+3: nobody reads them now)
    if (tid == nth - 1) {
      if (q + 3 < a.nRows) meta[(q + 3) & 3].i = pfI;
      if (q + 2 < a.nRows) {
        SgdPipeMeta &m2 = meta[(q + 2) & 3];
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
    __syncthreads();
    if (a.nFields == -7 && tid == 0) {   // phase profile (debug): cycles of this sample's phases
      long long c4 = clock64();
      prof[0] += c1 - c0; prof[1] += c2 - c1; prof[2] += c3 - c2; prof[3] += c4 - c3;
    }
    // ---- resetScaling (sgd.nim:116-131)
    const bool resetW = a.fitLinear && nscW < 1e-9, resetP = nscP < 1e-9;
    if (resetW || resetP) {
      sgd_materialize(a, SB8, a.d, resetW, resetP, nscP, nscW);
      if (tid == 0) {
        if (resetW) sh[2] = 1.0;
        if (resetP) sh[1] = 1.0;
      }
      __syncthreads();
    }
  }
  if (a.nFields == -7 && tid == 0)
    printf("[sgd pipe profile] cycles/sample: loads %lld  scale+forward %lld  reduce+loss %lld  update+park %lld\n",
           prof[0] / a.nRows, prof[1] / a.nRows, prof[2] / a.nRows, prof[3] / a.nRows);
  viol = block_sum(viol, red);
  __syncthreads();
  lossAcc = block_sum(lossAcc, red);
  if (tid == 0) {
    a.scal[0] = sh[1];
    a.scal[1] = sh[2];
    a.scal[2] = viol;
    a.scal[3] = lossAcc;
  }
}

// finalize (sgd.nim:99-113)
template <bool FFM>
__global__ void __launch_bounds__(SGD_THREADS, 1) sgd_finalize_kernel(const SgdArgs a) {
  const int SB8 = (FFM ? a.nFields : a.nOrders) * a.k;
  const double scP = a.scal[0], scW = a.scal[1];
  __syncthreads();
  if (a.fitLinear) {
    for (int64_t j = threadIdx.x; j < a.d; j += blockDim.x) {
      double v = a.w[j] * scW;
      a.w[j] = v / a.scalingsW[j];
      a.scalingsW[j] = 1.0;
    }
  }
  for (int64_t e = threadIdx.x; e < a.dd * SB8; e += blockDim.x) a.P[e] *= scP / a.scalingsP[e / SB8];
  __syncthreads();
  for (int64_t j = threadIdx.x; j < a.dd; j += blockDim.x) a.scalingsP[j] = 1.0;
  if (threadIdx.x == 0) {
    if (a.fitLinear) a.scal[1] = 1.0;
    a.scal[0] = 1.0;
  }
}

__global__ void sgd_fill_kernel(double *p, int64_t n, double v) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) p[e] = v;
}

template <class Model>
static int sgd_begin_common(nimfm_ctx *ctx, Model *m, int64_t dd, int64_t d) {
  CK(cudaSetDevice(ctx->device));
  if (!m->scalingsP) {
    CK(cudaMalloc(&m->scalingsP, (size_t)dd * 8));
    CK(cudaMalloc(&m->scalingsW, (size_t)d * 8));
    CK(cudaMalloc(&m->sgdScal, 8 * 8));
  }
  sgd_fill_kernel<<<64, 256, 0, ctx->stream>>>(m->scalingsP, dd, 1.0);   // sgd.nim:269-272
  sgd_fill_kernel<<<64, 256, 0, ctx->stream>>>(m->scalingsW, d, 1.0);
  ctx->launches += 2;
  const double sc[4] = {1.0, 1.0, 0.0, 0.0};
  CK(cudaMemcpyAsync(m->sgdScal, sc, 32, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  m->sgdReady = true;
  return NIMFM_OK;
}

extern "C" {

int32_t nimfm_fm_sgd_begin(nimfm_ctx *ctx, nimfm_fm *fm) {
  if (!ctx || !fm) return NIMFM_ERR_INVALID;
  return sgd_begin_common(ctx, fm, fm->dd(), fm->d);
}

int32_t nimfm_fm_sgd_epoch(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const nimfm_sgd_cfg *cfg,
                           int64_t *it, const int64_t *perm, int64_t nRows, double *viol, double *lossSum) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(fm && X && cfg && it, "NULL argument");
  if (!fm->sgdReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_fm_sgd_begin was not called");
  REQUIRE(X->kind != NIMFM_DS_CSC, "a CSR dataset is required");
  REQUIRE(X->d == fm->d, "Invalid nFeatures.");
  REQUIRE(X->y != nullptr, "dataset has no targets");
  REQUIRE(nRows >= 0 && (perm || nRows <= X->n), "bad nRows");
  CK(cudaSetDevice(ctx->device));
  int rc;
  const int32_t *permDev = nullptr;
  if (perm && nRows > 0) {
    if ((rc = nimfm_stage_row_ids(ctx, perm, nRows, X->n))) return rc;
    permDev = ctx->idx32Scratch;
  }
  SgdArgs a;
  memset(&a, 0, sizeof(a));
  a.data = X->data; a.indices = X->indices; a.indptr = X->indptr; a.y = X->y; a.perm = permDev;
  a.nRows = nRows; a.d = fm->d; a.dd = fm->dd();
  a.degree = fm->degree; a.k = fm->k; a.nOrders = fm->nOrders; a.nAug = fm->nAug;
  a.fitLinear = fm->fitLinear; a.fitIntercept = fm->fitIntercept;
  a.P = fm->P; a.w = fm->w; a.b = fm->b;
  a.scalingsP = fm->scalingsP; a.scalingsW = fm->scalingsW; a.scal = fm->sgdScal;
  a.cfg = *cfg; a.it0 = *it;
  // staged form when a row's slice fits shared memory and (order, component) fits one thread each
  const int SB8 = fm->nOrders * fm->k;
  const int zmax = (int)std::max<int64_t>(X->maxSegNnz + fm->nAug, 1);
  const size_t smem = ((size_t)zmax * SB8 + 3 * (size_t)zmax) * 8 + (size_t)zmax * 8;
  const char *env = getenv("NIMFM_SGD_KERNEL");
  const size_t smemPipe = ((size_t)zmax * SB8 + (size_t)SB8 * (NIMFM_MAX_DEGREE + 1) + 4 * (size_t)zmax) * 8 + 2 * (size_t)zmax * 4 + (size_t)SB8 + 16;
  // degree 1 (SB8 = 0, no P) runs the unstaged loop: its P passes are empty, the staged and pipelined forms divide by SB8
  if (SB8 == 0) {
    sgd_epoch_kernel<false><<<1, SGD_THREADS, 0, ctx->stream>>>(a);
  } else if (SB8 <= SGDP_THREADS - 64 && zmax <= 64 && (size_t)zmax * SB8 <= (size_t)SGDP_R * SGDP_THREADS && smemPipe <= (size_t)ctx->smemOptin - 4096 && !env) {
    if (getenv("NIMFM_SGD_PROFILE")) a.nFields = -7;
    CK(cudaFuncSetAttribute(sgd_fm_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smemPipe));
    sgd_fm_pipe_kernel<<<1, SGDP_THREADS, smemPipe, ctx->stream>>>(a, zmax);
  } else if (SB8 <= SGD_THREADS && smem <= (size_t)ctx->smemOptin - 2048 && !(env && !strcmp(env, "unstaged"))) {
    CK(cudaFuncSetAttribute(sgd_fm_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    sgd_fm_staged_kernel<<<1, SGD_THREADS, smem, ctx->stream>>>(a, zmax);
  } else {
    sgd_epoch_kernel<false><<<1, SGD_THREADS, 0, ctx->stream>>>(a);
  }
  LAUNCHED(ctx);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ctx->hostScalars, fm->sgdScal, 32, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *it += nRows;
  if (viol) *viol = ctx->hostScalars[2];
  if (lossSum) *lossSum = ctx->hostScalars[3];
  return NIMFM_OK;
}

int32_t nimfm_fm_sgd_end(nimfm_ctx *ctx, nimfm_fm *fm) {
  if (!ctx || !fm) return NIMFM_ERR_INVALID;
  if (!fm->sgdReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_fm_sgd_begin was not called");
  CK(cudaSetDevice(ctx->device));
  SgdArgs a;
  memset(&a, 0, sizeof(a));
  a.d = fm->d; a.dd = fm->dd(); a.k = fm->k; a.nOrders = fm->nOrders; a.fitLinear = fm->fitLinear;
  a.P = fm->P; a.w = fm->w; a.scalingsP = fm->scalingsP; a.scalingsW = fm->scalingsW; a.scal = fm->sgdScal;
  sgd_finalize_kernel<false><<<1, SGD_THREADS, 0, ctx->stream>>>(a);
  LAUNCHED(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  return NIMFM_OK;
}

int32_t nimfm_ffm_sgd_begin(nimfm_ctx *ctx, nimfm_ffm *m) {
  if (!ctx || !m) return NIMFM_ERR_INVALID;
  return sgd_begin_common(ctx, m, m->d, m->d);
}

int32_t nimfm_ffm_sgd_epoch(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, const nimfm_sgd_cfg *cfg,
                            int64_t *it, const int64_t *perm, int64_t nRows, double *viol, double *lossSum) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(m && X && cfg && it, "NULL argument");
  if (!m->sgdReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_ffm_sgd_begin was not called");
  REQUIRE(X->kind == NIMFM_DS_CSR_FIELD, "a CSRFieldDataset is required");
  REQUIRE(X->d == m->d, "Invalid nFeatures.");
  REQUIRE(X->nFields == m->nFields, "Invalid nFields.");
  REQUIRE(X->y != nullptr, "dataset has no targets");
  REQUIRE(nRows >= 0 && (perm || nRows <= X->n), "bad nRows");
  CK(cudaSetDevice(ctx->device));
  int rc;
  const int32_t *permDev = nullptr;
  if (perm && nRows > 0) {
    if ((rc = nimfm_stage_row_ids(ctx, perm, nRows, X->n))) return rc;
    permDev = ctx->idx32Scratch;
  }
  double *dA = nullptr;
  const size_t dAn = (size_t)std::max<int64_t>(X->maxSegNnz, 1) * m->nFields * m->k;
  CK(cudaMalloc(&dA, dAn * 8));
  SgdArgs a;
  memset(&a, 0, sizeof(a));
  a.data = X->data; a.indices = X->indices; a.fields = X->fields; a.indptr = X->indptr; a.y = X->y; a.perm = permDev;
  a.nRows = nRows; a.d = m->d; a.dd = m->d;
  a.k = m->k; a.nFields = (int)m->nFields;
  a.fitLinear = m->fitLinear; a.fitIntercept = m->fitIntercept;
  a.P = m->P; a.w = m->w; a.b = m->b;
  a.scalingsP = m->scalingsP; a.scalingsW = m->scalingsW; a.scal = m->sgdScal; a.dA = dA;
  a.cfg = *cfg; a.it0 = *it;
  sgd_epoch_kernel<true><<<1, SGD_THREADS, 0, ctx->stream>>>(a);
  LAUNCHED(ctx);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ctx->hostScalars, m->sgdScal, 32, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaFree(dA));
  *it += nRows;
  if (viol) *viol = ctx->hostScalars[2];
  if (lossSum) *lossSum = ctx->hostScalars[3];
  return NIMFM_OK;
}

int32_t nimfm_ffm_sgd_end(nimfm_ctx *ctx, nimfm_ffm *m) {
  if (!ctx || !m) return NIMFM_ERR_INVALID;
  if (!m->sgdReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_ffm_sgd_begin was not called");
  CK(cudaSetDevice(ctx->device));
  SgdArgs a;
  memset(&a, 0, sizeof(a));
  a.d = m->d; a.dd = m->d; a.k = m->k; a.nFields = (int)m->nFields; a.fitLinear = m->fitLinear;
  a.P = m->P; a.w = m->w; a.scalingsP = m->scalingsP; a.scalingsW = m->scalingsW; a.scal = m->sgdScal;
  sgd_finalize_kernel<true><<<1, SGD_THREADS, 0, ctx->stream>>>(a);
  LAUNCHED(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  return NIMFM_OK;
}

}  // extern "C"
