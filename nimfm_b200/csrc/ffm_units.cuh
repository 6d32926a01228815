// ffm_units.cuh -- (nonzero, field) FFM kernel (K10 / K11: decisionFunction, predict+grad, AdaGrad minibatch) for
// every nComponents and row length: the route for the shapes the staged ffm_rows_kernel cannot hold in shared memory.
//
// ONE THREAD BLOCK PER ROW.  The block sorts the row's {x, j, f} records by field and lists the row's non-empty field
// buckets (at most z of them, nothing sized by nFields).  One UNIT is a (nonzero u, non-empty bucket f) pair; a group
// of KT lanes evaluates it by coalesced gathers from the P[j][f][s] layout:
//     acc[s] = sum_{v in bucket f, v != u, j_v != j_u} x_v * P[j_v][f_u][s]          (sgd_ffm.nim:23-30)
// forward   yhat = b + lin + 1/2 sum_{u,f} x_u <P[j_u][f][:], acc>   (every pair counted once from each side)
// backward  g[j_u][f][s] += coef * x_u * acc[s]   (acc recomputed; its gathers hit L2)
// acc is the sample's whole gradient entry, so AdaGrad's square (adagrad.nim:119-124) is exact when fields repeat in
// a row.  Shared memory holds only the row's records and bucket bounds: 20 B per nonzero, independent of nFields * k.
//
// k is a run-time value: lanes with s >= k idle, and a group loops over KT-wide chunks of s.  Element offsets are
// 64-bit, so d * nFields >= 2^31 is served.  Rows of up to FFM_UNITS_SMEM_CAP nonzeros are bucketed in shared memory;
// a longer row uses the block's slice of a global scratch area of the same layout (FfmArgs::unitScratch,
// ffm_units_row_bytes(CH) bytes per block, owned by the model).
#pragma once
#include "common.cuh"

#define FFM_UNITS_THREADS 256
#define FFM_UNITS_SMEM_CAP 2048   // rows up to this many nonzeros are bucketed in shared memory (40 KB)

// bytes one row of up to `cap` nonzeros needs: cap records + cap + 1 bucket bounds
__host__ __device__ inline size_t ffm_units_row_bytes(int64_t cap) {
  return ((size_t)cap * sizeof(FfmMeta) + (size_t)(cap + 1) * sizeof(int) + 15) & ~(size_t)15;
}

template <int MODE, int KT>
__global__ void __launch_bounds__(FFM_UNITS_THREADS, 4) ffm_units_kernel(const FfmArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double red[FFM_UNITS_THREADS / 32];
  __shared__ double shv;
  __shared__ int shNb;
  const int k = a.k, nF = a.nFields;
  const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31;
  const int sl = tid & (KT - 1), grp = tid / KT, nGrp = nth / KT;
  const int capS = a.CH < FFM_UNITS_SMEM_CAP ? a.CH : FFM_UNITS_SMEM_CAP;
  double accLoss = 0.0, accB1 = 0.0, accB2 = 0.0;
  double bias = a.b[0];
  if (MODE == FFM_ADAGRAD && !a.first && a.fitIntercept)   // adagrad.nim:101-105 (batch snapshot)
    bias = -a.eta0 * a.adaScal[0] / (sqrt(a.adaScal[1]) + a.eta0 * a.tIt * a.alpha0);

  for (int64_t q = blockIdx.x; q < a.nRows; q += gridDim.x) {
    const int64_t r = a.rowIdx ? (int64_t)a.rowIdx[q] : (a.rowBegin + q) % a.n;
    const int64_t rb = a.indptr[r];
    const int z = (int)(a.indptr[r + 1] - rb);
    unsigned char *base = z <= capS ? smem_raw : a.unitScratch + (size_t)blockIdx.x * ffm_units_row_bytes(a.CH);
    FfmMeta *rec = reinterpret_cast<FfmMeta *>(base);
    int *bnd = reinterpret_cast<int *>(rec + z);   // [z + 1]: the row's fields, then the bucket bounds
    __syncthreads();                               // the previous row's records are no longer read
    double lin = 0.0;
    for (int u = tid; u < z; u += nth) {
      bnd[u] = a.fields[rb + u];
      lin += a.w[a.indices[rb + u]] * a.data[rb + u];
    }
    __syncthreads();
    // ---- records sorted by (field, position): rank counting, O(z^2 / threads) like the unit loop itself
    for (int u = tid; u < z; u += nth) {
      const int f = bnd[u];
      int rank = 0;
      for (int v = 0; v < z; ++v) {
        const int fv = bnd[v];
        rank += (fv < f) | ((fv == f) & (v < u));
      }
      FfmMeta m;
      m.x = a.data[rb + u];
      m.j = a.indices[rb + u];
      m.f = f;
      rec[rank] = m;
    }
    __syncthreads();
    // ---- compact list of the non-empty buckets: bnd[b] = first sorted position of bucket b, bnd[nb] = z
    if (tid < 32) {
      int carry = 0;
      for (int p0 = 0; p0 < z; p0 += 32) {
        const int p = p0 + lane;
        const bool start = p < z && (p == 0 || rec[p].f != rec[p - 1].f);
        const unsigned msk = __ballot_sync(0xffffffffu, start);
        if (start) bnd[carry + __popc(msk & ((1u << lane) - 1u))] = p;
        carry += __popc(msk);
      }
      if (lane == 0) {
        bnd[carry] = z;
        shNb = carry;
      }
    }
    __syncthreads();
    const int nb = shNb;
    // units e = u * nb + b, dealt to the groups round-robin; (u, b) advances by nGrp without a division
    const int du = nb ? nGrp / nb : 0, db = nb ? nGrp % nb : 0;
    const int64_t nUnits = (int64_t)z * nb;

    // ---- forward
    double part = 0.0;
    {
      int u = nb ? grp / nb : 0, b = nb ? grp % nb : 0;
      for (int64_t e = grp; e < nUnits; e += nGrp) {
        const FfmMeta mu = rec[u];
        const int t0 = bnd[b], t1 = bnd[b + 1];
        const int f = rec[t0].f;
        const double *Pu = a.P + ((int64_t)mu.j * nF + f) * k;
        for (int s = sl; s < k; s += KT) {
          double acc = 0.0;
          for (int t = t0; t < t1; ++t) {
            const FfmMeta mv = rec[t];
            if (t != u && mv.j != mu.j) acc += mv.x * __ldg(a.P + ((int64_t)mv.j * nF + mu.f) * k + s);
          }
          part += __ldg(Pu + s) * (mu.x * acc);
        }
        u += du;
        b += db;
        if (b >= nb) { b -= nb; ++u; }
      }
    }
    const double tot = block_sum(lin + 0.5 * part, red);
    if (tid == 0) {
      const double yhat = bias + tot;
      if (a.yOut) a.yOut[q] = yhat;
      if (MODE != FFM_PREDICT) {
        const double yi = a.y[r];
        const double dL = dev_dloss(a.loss, a.thr, yi, yhat);
        accLoss += dev_loss(a.loss, a.thr, yi, yhat);
        const double coef = MODE == FFM_GRAD ? dL / a.mb : dL;
        accB1 += coef;
        accB2 += dL * dL;
        shv = coef;
      }
    }
    if (MODE == FFM_PREDICT) continue;
    __syncthreads();
    const double coef = shv;

    // ---- backward: one gradient entry (j_u, f) per unit
    {
      int u = nb ? grp / nb : 0, b = nb ? grp % nb : 0;
      for (int64_t e = grp; e < nUnits; e += nGrp) {
        const FfmMeta mu = rec[u];
        const int t0 = bnd[b], t1 = bnd[b + 1];
        const int64_t ge = ((int64_t)mu.j * nF + rec[t0].f) * k;
        for (int s = sl; s < k; s += KT) {
          double acc = 0.0;
          for (int t = t0; t < t1; ++t) {
            const FfmMeta mv = rec[t];
            if (t != u && mv.j != mu.j) acc += mv.x * __ldg(a.P + ((int64_t)mv.j * nF + mu.f) * k + s);
          }
          const double gr = coef * (mu.x * acc);
          if (gr != 0.0) {
            atomicAdd(a.gP + ge + s, gr);
            if (MODE == FFM_ADAGRAD) atomicAdd(a.dGnP + ge + s, gr * gr);
          }
        }
        u += du;
        b += db;
        if (b >= nb) { b -= nb; ++u; }
      }
    }
    if (a.fitLinear)
      for (int u = tid; u < z; u += nth) {
        const FfmMeta m = rec[u];
        const double gx = coef * m.x;
        atomicAdd(a.gw + m.j, gx);
        if (MODE == FFM_ADAGRAD) atomicAdd(a.dGnw + m.j, gx * gx);
      }
  }
  if (MODE != FFM_PREDICT && tid == 0) {
    a.partials[blockIdx.x * 4 + 0] = accLoss;
    a.partials[blockIdx.x * 4 + 1] = accB1;
    a.partials[blockIdx.x * 4 + 2] = accB2;
    a.partials[blockIdx.x * 4 + 3] = 0.0;
  }
}
