// ffm_pairs.cuh -- pair-streaming FFM kernel (K10 / K11: decisionFunction, predict+grad, AdaGrad
// minibatch) for nComponents KT in {4, 8, 16, 32}: ONE WARP PER ROW, 32/KT "pair slots" of KT lanes each.
//
// It follows the reference's own loop (field_aware_factorization_machine.nim:68-76, sgd_ffm.nim:23-30):
// for every unordered pair of the row's nonzeros (u, v),
//     yhat      += x_u x_v <P[j_u][f_v][:], P[j_v][f_u][:]>
//     dA[f_v][j_u][:] += x_u x_v P[j_v][f_u][:]      dA[f_u][j_v][:] += x_u x_v P[j_u][f_v][:]
// The z(z-1)/2 pairs of a row are enumerated by ONE linear index (slot s takes pairs s, s+SLOTS, ...),
// so every slot has the same trip count, and they are processed PB at a time: the 2*PB gathers of a
// batch (each a coalesced KT*8-byte segment of the P[j][f][s] layout) are all issued before the first
// is consumed.  ncu on the previous form (2 pairs in flight, r01g): issue slots 16 % busy,
// long_scoreboard 20 warps per issue -- purely latency-bound on its own gathers with DRAM at 22 %.
// The backward pass re-loads the two vectors (mostly L2 hits) and emits both gradient vectors with
// FP64 RED atomics; AdaGrad also emits their squares (valid because the AdaGrad route is only taken
// for datasets with at most one nonzero per (row, field), where a pair's contribution IS the sample's
// whole gradient entry -- adagrad.nim:119-124 squares the per-sample gradient).
// Nothing is staged in shared memory except the row's {x, j, f} records, so occupancy is
// register-bound (vs 2 rows/SM for the block-per-row kernel in ffm.cu, the general fallback).
#pragma once
#include "common.cuh"

struct FfmArgs;   // defined in ffm.cu

struct __align__(16) FfmRec {
  double x;
  int32_t jb;   // j * nFields: (jb + f) * k is the element offset of P[j][f][0]  (d * nFields < 2^31 is required)
  int32_t f;
};

enum { FFM_PAIRS_PREDICT = 0, FFM_PAIRS_GRAD = 1, FFM_PAIRS_ADAGRAD = 2 };
#define FFM_PAIRS_TABLE_MAXZ 64   // rows up to this length enumerate their pairs through a shared-memory table

// advance the pair cursor (u, v), u < v < z, by `step` positions of the row-major pair order
__device__ __forceinline__ void ffm_pair_advance(int &u, int &v, int step, int z) {
  v += step;
  while (v >= z && u < z - 1) {
    v = v - z + u + 2;
    u += 1;
  }
}

// bytes of shared memory one row needs: its records + (table) the pair table of the longest row
__host__ __device__ inline size_t ffm_pairs_warp_smem(int CH, bool table) {
  size_t b = (size_t)CH * sizeof(FfmRec) + (table ? (size_t)CH * (CH - 1) / 2 * sizeof(uint16_t) : 0);
  return (b + 15) & ~(size_t)15;
}

// The warp form runs the rows longer than FFM_PAIRS_TABLE_MAXZ (up to 1024 nonzeros), whose pair table would not
// fit: each slot walks the row-major pair order with a cursor (ffm_pair_advance).
template <int MODE, int KT, class Args>
__global__ void __launch_bounds__(256, 2) ffm_pairs_kernel(const Args a) {
  constexpr int SLOTS = 32 / KT;
  constexpr int PB = 8;   // pairs in flight per slot (2*PB gathers per lane)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  const int warpInBlock = threadIdx.x >> 5;
  const int s = lane & (KT - 1);
  const int slot = lane / KT;
  const int CH = a.CH;
  FfmRec *rec = reinterpret_cast<FfmRec *>(smem_raw + (size_t)warpInBlock * ffm_pairs_warp_smem(CH, false));
  const int warpsPerBlock = blockDim.x >> 5;
  const int64_t warpGlobal = (int64_t)blockIdx.x * warpsPerBlock + warpInBlock;
  const int64_t nWarps = (int64_t)gridDim.x * warpsPerBlock;
  const int nF = a.nFields;
  double bias = a.b[0];
  if (MODE == FFM_PAIRS_ADAGRAD && !a.first && a.fitIntercept)   // adagrad.nim:101-105 (batch snapshot)
    bias = -a.eta0 * a.adaScal[0] / (sqrt(a.adaScal[1]) + a.eta0 * a.tIt * a.alpha0);
  const double *__restrict__ Pg = a.P + s;
  double accLoss = 0.0, accB1 = 0.0, accB2 = 0.0;

  for (int64_t q = warpGlobal; q < a.nRows; q += nWarps) {
    const int64_t r = a.rowIdx ? (int64_t)a.rowIdx[q] : (a.rowBegin + q) % a.n;
    const int64_t rb = a.indptr[r];
    const int z = (int)(a.indptr[r + 1] - rb);
    __syncwarp();
    double lin = 0.0;
    for (int u = lane; u < z; u += 32) {
      FfmRec m;
      const int32_t j = a.indices[rb + u];
      m.jb = j * nF;
      m.f = a.fields[rb + u];
      m.x = a.data[rb + u];
      rec[u] = m;
      lin += a.w[j] * m.x;
    }
    const int nPairs = z * (z - 1) / 2;
    __syncwarp();

    // ---- forward: running dot over this slot's pairs
    double acc = 0.0;
    {
      int u = 0, v = 1;
      ffm_pair_advance(u, v, slot, z);
      for (int p = slot; p < nPairs; p += SLOTS * PB) {
        double a1[PB], a2[PB], xx[PB];
#pragma unroll
        for (int i = 0; i < PB; ++i) {
          const bool ok = p + i * SLOTS < nPairs;
          a1[i] = 0.0; a2[i] = 0.0; xx[i] = 0.0;
          if (ok) {
            const FfmRec mu = rec[u], mv = rec[v];
            if (mv.jb != mu.jb) {                                               // the reference pairs j1 < j2 only
              a1[i] = __ldg(Pg + (int64_t)(mu.jb + mv.f) * KT);                 // P[j_u][f_v][s]
              a2[i] = __ldg(Pg + (int64_t)(mv.jb + mu.f) * KT);                 // P[j_v][f_u][s]
              xx[i] = mu.x * mv.x;
            }
          }
          ffm_pair_advance(u, v, SLOTS, z);
        }
#pragma unroll
        for (int i = 0; i < PB; ++i) acc += xx[i] * (a1[i] * a2[i]);
      }
    }
    const double yhat = bias + warp_sum(lin + acc);
    if (lane == 0 && a.yOut) a.yOut[q] = yhat;
    if (MODE == FFM_PAIRS_PREDICT) continue;

    const double yi = a.y[r];
    const double dL = dev_dloss(a.loss, a.thr, yi, yhat);
    const double coef = (MODE == FFM_PAIRS_GRAD) ? dL / a.mb : dL;
    if (lane == 0) {
      accLoss += dev_loss(a.loss, a.thr, yi, yhat);
      accB1 += coef;
      accB2 += dL * dL;
    }
    // ---- backward: both gradient vectors of every pair
    double *__restrict__ gPg = a.gP + s;
    double *__restrict__ gNg = (MODE == FFM_PAIRS_ADAGRAD) ? a.dGnP + s : nullptr;
    {
      int u = 0, v = 1;
      ffm_pair_advance(u, v, slot, z);
      for (int p = slot; p < nPairs; p += SLOTS * PB) {
        double a1[PB], a2[PB], cx[PB];
        int32_t e1[PB], e2[PB];   // (j*nFields + f): element offset / KT
#pragma unroll
        for (int i = 0; i < PB; ++i) {
          const bool ok = p + i * SLOTS < nPairs;
          e1[i] = -1; e2[i] = 0; a1[i] = 0.0; a2[i] = 0.0; cx[i] = 0.0;
          if (ok) {
            const FfmRec mu = rec[u], mv = rec[v];
            if (mv.jb != mu.jb) {
              e1[i] = mu.jb + mv.f;                        // entry (j_u, f_v)
              e2[i] = mv.jb + mu.f;                        // entry (j_v, f_u)
              a1[i] = __ldg(Pg + (int64_t)e1[i] * KT);
              a2[i] = __ldg(Pg + (int64_t)e2[i] * KT);
              cx[i] = coef * (mu.x * mv.x);
            }
          }
          ffm_pair_advance(u, v, SLOTS, z);
        }
#pragma unroll
        for (int i = 0; i < PB; ++i) {
          if (e1[i] >= 0) {
            const double g1 = cx[i] * a2[i], g2 = cx[i] * a1[i];
            atomicAdd(gPg + (int64_t)e1[i] * KT, g1);
            atomicAdd(gPg + (int64_t)e2[i] * KT, g2);
            if (MODE == FFM_PAIRS_ADAGRAD) {
              atomicAdd(gNg + (int64_t)e1[i] * KT, g1 * g1);
              atomicAdd(gNg + (int64_t)e2[i] * KT, g2 * g2);
            }
          }
        }
      }
    }
    if (a.fitLinear)
      for (int u = lane; u < z; u += 32) {
        const double gx = coef * rec[u].x;
        const int32_t j = a.indices[rb + u];
        atomicAdd(a.gw + j, gx);
        if (MODE == FFM_PAIRS_ADAGRAD) atomicAdd(a.dGnw + j, gx * gx);
      }
  }
  if (MODE != FFM_PAIRS_PREDICT) {
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

// ------------------------------------------------------------------ block-per-row form of the same loop
// ONE THREAD BLOCK PER ROW: the row's pairs are dealt to all (blockDim/32)*SLOTS pair slots of the block,
// so a 39-nonzero row is 3 batches of 8 pairs per slot instead of 24.  Only gridDim rows are in flight
// on the chip (296 x 95 KB of gathered parameters ~ 28 MB), so the backward pass's re-read of the row's
// vectors and the second half of every 128-byte line (the neighbouring field's vector) hit L2; with a
// warp per row 2 368 rows x 95 KB = 225 MB are in flight, more than the 126 MB L2 (ncu r01i: 130 KB/row of
// DRAM reads for 95 KB of algorithmic gathers, DRAM the only unit above 30 %).
// Requires z <= FFM_PAIRS_TABLE_MAXZ (the shared pair table); summation order differs from the warp
// form only by association.
//
// BULK (gradient modes; datasets without repeated fields in a row): the backward pass is organised by NONZERO
// instead of by pair.  In the P[j][f][s] layout the gradient of nonzero u is ONE contiguous block of
// nFields*k doubles, g[j_u][f_v][:] = coef x_u x_v P[j_v][f_u][:] over the row's other nonzeros v.  A warp
// builds that block in shared memory (one coalesced k*8-byte gather and one shared-memory store per partner)
// and hands it to the TMA unit as one `cp.reduce.async.bulk.global.shared::cta.add.f64` (SASS UBLKRED.G.S.ADD.F64)
// -- 39 bulk reductions of 2 496 B per C5 row instead of 370 warp-wide REDs touching four 64-byte segments each.
// scratch/red_rate.cu: the L2 adds FP64 at the same ~4.7 TB/s either way when the lines are resident, but on lines
// that miss, 64-byte RED segments reach 1.36 TB/s and 2 KB bulk reductions 2.78 TB/s.
__host__ __device__ inline size_t ffm_bulk_stage_off(int CH) { return (ffm_pairs_warp_smem(CH, true) + 127) & ~(size_t)127; }
__host__ __device__ inline size_t ffm_bulk_smem(int CH, int segDoubles, int nAcc, int warps) {
  return ffm_bulk_stage_off(CH) + (size_t)warps * 2 * nAcc * segDoubles * 8;
}

template <int MODE, int KT, class Args, bool BULK = false>
__global__ void __launch_bounds__(256, 2) ffm_pairs_block_kernel(const Args a) {
  constexpr int SLOTS = 32 / KT;
  constexpr int PB = 8;
  constexpr int PBK = 10;                                       // BULK: partners in flight per slot
  constexpr int NACC = (MODE == FFM_PAIRS_ADAGRAD) ? 2 : 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double red[32];
  const int lane = threadIdx.x & 31;
  const int warpInBlock = threadIdx.x >> 5;
  const int nWarpsB = blockDim.x >> 5;
  const int s = lane & (KT - 1);
  const int gslot = warpInBlock * SLOTS + lane / KT;
  const int nSlots = nWarpsB * SLOTS;
  const int CH = a.CH;
  FfmRec *rec = reinterpret_cast<FfmRec *>(smem_raw);
  uint16_t *tab = reinterpret_cast<uint16_t *>(smem_raw + (size_t)CH * sizeof(FfmRec));
  int zTab = -1;
  const int nF = a.nFields;
  double bias = a.b[0];
  if (MODE == FFM_PAIRS_ADAGRAD && !a.first && a.fitIntercept)
    bias = -a.eta0 * a.adaScal[0] / (sqrt(a.adaScal[1]) + a.eta0 * a.tIt * a.alpha0);
  const double *__restrict__ Pg = a.P + s;
  double accLoss = 0.0, accB1 = 0.0, accB2 = 0.0;
  const int segD = nF * KT;                                      // doubles of one feature's block
  double *stage = reinterpret_cast<double *>(smem_raw + ffm_bulk_stage_off(CH)) + (size_t)warpInBlock * 2 * NACC * segD;
  int bulkIt = 0;                                                // per warp: which of its two stage buffers is next

  for (int64_t q = blockIdx.x; q < a.nRows; q += gridDim.x) {
    const int64_t r = a.rowIdx ? (int64_t)a.rowIdx[q] : (a.rowBegin + q) % a.n;
    const int64_t rb = a.indptr[r];
    const int z = (int)(a.indptr[r + 1] - rb);
    __syncthreads();                                   // the previous row's records are no longer read
    double lin = 0.0;
    for (int u = threadIdx.x; u < z; u += blockDim.x) {
      FfmRec m;
      const int32_t j = a.indices[rb + u];
      m.jb = j * nF;
      m.f = a.fields[rb + u];
      m.x = a.data[rb + u];
      rec[u] = m;
      lin += a.w[j] * m.x;
    }
    const int nPairs = z * (z - 1) / 2;
    if (z != zTab) {
      int u = 0, v = 1;
      ffm_pair_advance(u, v, threadIdx.x, z);
      for (int p = threadIdx.x; p < nPairs; p += blockDim.x) {
        tab[p] = (uint16_t)(u | (v << 8));
        ffm_pair_advance(u, v, blockDim.x, z);
      }
      zTab = z;
    }
    __syncthreads();

    // ---- forward
    double acc = 0.0;
    for (int p = gslot; p < nPairs; p += nSlots * PB) {
      double a1[PB], a2[PB], xx[PB];
#pragma unroll
      for (int i = 0; i < PB; ++i) {
        const int pi = p + i * nSlots;
        a1[i] = 0.0; a2[i] = 0.0; xx[i] = 0.0;
        if (pi < nPairs) {
          const unsigned uv = tab[pi];
          const FfmRec mu = rec[uv & 0xff], mv = rec[uv >> 8];
          if (mv.jb != mu.jb) {
            a1[i] = __ldg(Pg + (int64_t)(mu.jb + mv.f) * KT);
            a2[i] = __ldg(Pg + (int64_t)(mv.jb + mu.f) * KT);
            xx[i] = mu.x * mv.x;
          }
        }
      }
#pragma unroll
      for (int i = 0; i < PB; ++i) acc += xx[i] * (a1[i] * a2[i]);
    }
    double part = warp_sum(lin + acc);
    if (lane == 0) red[warpInBlock] = part;
    __syncthreads();
    double tot = 0.0;
    for (int wq = 0; wq < nWarpsB; ++wq) tot += red[wq];   // fixed order, identical in every thread
    const double yhat = bias + tot;
    if (threadIdx.x == 0 && a.yOut) a.yOut[q] = yhat;
    if (MODE == FFM_PAIRS_PREDICT) continue;

    const double yi = a.y[r];
    const double dL = dev_dloss(a.loss, a.thr, yi, yhat);
    const double coef = (MODE == FFM_PAIRS_GRAD) ? dL / a.mb : dL;
    if (threadIdx.x == 0) {
      accLoss += dev_loss(a.loss, a.thr, yi, yhat);
      accB1 += coef;
      accB2 += dL * dL;
    }
    // ---- backward
    double *__restrict__ gPg = a.gP + s;
    double *__restrict__ gNg = (MODE == FFM_PAIRS_ADAGRAD) ? a.dGnP + s : nullptr;
    if (BULK) {
      const int slotW = lane / KT;
      for (int u = warpInBlock; u < z; u += nWarpsB, ++bulkIt) {
        double *sb = stage + (size_t)(bulkIt & 1) * NACC * segD;
        // the bulk reduction issued two iterations ago has finished READING this buffer
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncwarp();
        const FfmRec mu = rec[u];
        if (z != nF) {                                           // absent fields contribute nothing
          for (int e = lane; e < NACC * segD; e += 32) sb[e] = 0.0;
          __syncwarp();
        }
        for (int v0 = slotW; v0 < z; v0 += SLOTS * PBK) {
          double a2[PBK], cx[PBK];
          int32_t fv[PBK];
#pragma unroll
          for (int i = 0; i < PBK; ++i) {
            const int v = v0 + i * SLOTS;
            fv[i] = -1; a2[i] = 0.0; cx[i] = 0.0;
            if (v < z) {
              const FfmRec mv = rec[v];
              fv[i] = mv.f;
              if (mv.jb != mu.jb) {                              // v == u (or the same feature again): a zero segment
                a2[i] = __ldg(Pg + (int64_t)(mv.jb + mu.f) * KT);   // P[j_v][f_u][s]
                cx[i] = coef * (mu.x * mv.x);
              }
            }
          }
#pragma unroll
          for (int i = 0; i < PBK; ++i) {
            if (fv[i] >= 0) {
              const double g = cx[i] * a2[i];
              sb[fv[i] * KT + s] = g;                            // entry (j_u, f_v)
              if (MODE == FFM_PAIRS_ADAGRAD) sb[segD + fv[i] * KT + s] = g * g;
            }
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          const uint32_t bytes = (uint32_t)segD * 8u;
          const uint32_t src = (uint32_t)__cvta_generic_to_shared(sb);
          asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f64 [%0], [%1], %2;"
                       ::"l"(a.gP + (int64_t)mu.jb * KT), "r"(src), "r"(bytes) : "memory");
          if (MODE == FFM_PAIRS_ADAGRAD)
            asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f64 [%0], [%1], %2;"
                         ::"l"(a.dGnP + (int64_t)mu.jb * KT), "r"(src + bytes), "r"(bytes) : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
      }
    } else
    for (int p = gslot; p < nPairs; p += nSlots * PB) {
      double a1[PB], a2[PB], cx[PB];
      int32_t e1[PB], e2[PB];
#pragma unroll
      for (int i = 0; i < PB; ++i) {
        const int pi = p + i * nSlots;
        e1[i] = -1; e2[i] = 0; a1[i] = 0.0; a2[i] = 0.0; cx[i] = 0.0;
        if (pi < nPairs) {
          const unsigned uv = tab[pi];
          const FfmRec mu = rec[uv & 0xff], mv = rec[uv >> 8];
          if (mv.jb != mu.jb) {
            e1[i] = mu.jb + mv.f;
            e2[i] = mv.jb + mu.f;
            a1[i] = __ldg(Pg + (int64_t)e1[i] * KT);
            a2[i] = __ldg(Pg + (int64_t)e2[i] * KT);
            cx[i] = coef * (mu.x * mv.x);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < PB; ++i) {
        if (e1[i] >= 0) {
          const double g1 = cx[i] * a2[i], g2 = cx[i] * a1[i];
          atomicAdd(gPg + (int64_t)e1[i] * KT, g1);
          atomicAdd(gPg + (int64_t)e2[i] * KT, g2);
          if (MODE == FFM_PAIRS_ADAGRAD) {
            atomicAdd(gNg + (int64_t)e1[i] * KT, g1 * g1);
            atomicAdd(gNg + (int64_t)e2[i] * KT, g2 * g2);
          }
        }
      }
    }
    if (a.fitLinear)
      for (int u = threadIdx.x; u < z; u += blockDim.x) {
        const double gx = coef * rec[u].x;
        const int32_t j = a.indices[rb + u];
        atomicAdd(a.gw + j, gx);
        if (MODE == FFM_PAIRS_ADAGRAD) atomicAdd(a.dGnw + j, gx * gx);
      }
  }
  if (BULK && lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  if (MODE != FFM_PAIRS_PREDICT && threadIdx.x == 0) {
    a.partials[blockIdx.x * 4 + 0] = accLoss;
    a.partials[blockIdx.x * 4 + 1] = accB1;
    a.partials[blockIdx.x * 4 + 2] = accB2;
    a.partials[blockIdx.x * 4 + 3] = 0.0;
  }
}

// flag <- 1 if any row has two nonzeros of the same field (warp per row; the AdaGrad pair route needs 0)
static __global__ void ffm_field_dup_kernel(const int32_t *fields, const int64_t *indptr, int64_t n, int *flag) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nWarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp; r < n; r += nWarps) {
    const int64_t b = indptr[r], e = indptr[r + 1];
    for (int64_t u = b + lane; u < e; u += 32) {
      const int32_t f = fields[u];
      for (int64_t v = u + 1; v < e; ++v)
        if (fields[v] == f) *flag = 1;
    }
  }
}
