// fm_rows_stream.cuh -- register-streaming instance of the row kernel (K1 / K2) for the BASELINE
// shapes: nComponents KT in {8, 16, 32} fixed at compile time, degree 2 or 3, rows of at most CH
// nonzeros (CH <= 512).
//
// ncu on the shared-memory-staged kernels (profiles/r01_ncu_*fast*): 8-10 resident warps/SM (the
// 20-29 KB/row staging buffer is the occupancy limiter), issue slots 25 % busy, stalls dominated by
// long_scoreboard -- the kernel waits on its own gathers.  This instance trades the staging buffer for
// occupancy: the row's P slice is NOT staged; each lane streams its component's values through
// registers, U nonzeros x nOrders loads in flight per lane (coalesced KT*8-byte segments per load),
// the forward DP consumes them, and the backward pass re-gathers the same lines (L1/L2 hits: the row
// was just read) instead of re-reading shared memory.  Shared memory holds only the per-nonzero
// records {x, j, hot-slot offset} (16 B each) and the hot-column accumulators, so 20+ warps/SM fit.
// Arithmetic and summation structure are those of the generic kernel (fm_rows.cuh).
#pragma once
#include "fm_rows.cuh"

// one nonzero of the row: one LDS.128 per nonzero in the inner loops, no integer address math
struct __align__(16) NnzMeta {
  double x;
  int32_t j;
  int32_t acc;   // element offset of the hot-slot accumulator row in sAcc, or -1 (cold)
};

__host__ __device__ inline size_t stream_group_smem(int CH, int SB8, int nHotTot, int nAcc) {
  size_t b = (size_t)CH * sizeof(NnzMeta) + (size_t)nHotTot * (SB8 + 1) * 8 * (nAcc > 0 ? nAcc : 1);
  return (b + 15) & ~(size_t)15;
}

template <int DEGREE, bool EXPLICIT, int MODE, int KT>
__global__ void __launch_bounds__(256, (RowCfg<DEGREE, EXPLICIT>::NO == 1 || MODE == MODE_PREDICT) ? 4 : 2) fm_rows_stream_kernel(const RowArgs a) {
  // MODE_ADAGRAD = MODE_GRAD with coef = dloss (adagrad.nim:113-124) and a second scatter of the
  // squared gradient into the g_norm delta block; P was refreshed by adagrad_refresh_kernel.
  constexpr int NACC = (MODE == MODE_ADAGRAD) ? 2 : 1;
  constexpr int NO = RowCfg<DEGREE, EXPLICIT>::NO;
  constexpr int G = KT;
  constexpr int GPW = 32 / G;
  constexpr int SB8 = NO * KT;
  constexpr int ASTR = SB8 + 1;
  constexpr int U = 8;   // nonzeros in flight per lane
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  const int warpInBlock = threadIdx.x >> 5;
  const int gl = lane & (G - 1);
  const int gidInWarp = lane / G;
  const int CH = a.CH;
  const int nHotTot = (MODE == MODE_PREDICT || MODE == MODE_STASH) ? 0 : a.nHot + a.nAug;
  const size_t perGroup = stream_group_smem(CH, SB8, nHotTot, NACC);
  unsigned char *base = smem_raw + (size_t)(warpInBlock * GPW + gidInWarp) * perGroup;
  NnzMeta *sMeta = reinterpret_cast<NnzMeta *>(base);
  double *sAcc = reinterpret_cast<double *>(sMeta + CH);
  double *sAccN = sAcc + (size_t)nHotTot * ASTR;   // AdaGrad only
  for (int e = gl; e < nHotTot * ASTR * NACC; e += G) sAcc[e] = 0.0;
  __syncwarp();

  const int warpsPerBlock = blockDim.x >> 5;
  const int64_t warpGlobal = (int64_t)blockIdx.x * warpsPerBlock + warpInBlock;
  const int64_t nWarps = (int64_t)gridDim.x * warpsPerBlock;
  const int64_t tiles = (a.nRows + GPW - 1) / GPW;
  double accLoss = 0.0, accB1 = 0.0, accB2 = 0.0;
  double bias = a.b[0];
  if (MODE == MODE_ADAGRAD && !a.first && a.fitIntercept)   // the intercept every row of the batch sees
    bias = -a.eta0 * a.adaScal[0] / (sqrt(a.adaScal[1]) + a.eta0 * a.tIt * a.alpha0);
  const double *__restrict__ Pg = a.P + gl;

  for (int64_t tile = warpGlobal; tile < tiles; tile += nWarps) {
    const int64_t q = tile * GPW + gidInWarp;
    const bool active = q < a.nRows;
    int64_t r = 0;
    if (active) r = a.rowIdx ? (int64_t)a.rowIdx[q] : (a.rowBegin + q) % a.n;
    const int64_t rb = active ? a.indptr[r] : 0;
    const int zReal = active ? (int)(a.indptr[r + 1] - rb) : 0;
    const int z = active ? zReal + a.nAug : 0;
    int zmax = z;
    if (GPW > 1) {
#pragma unroll
      for (int off = 16; off >= G; off >>= 1) zmax = max(zmax, __shfl_xor_sync(0xffffffffu, zmax, off));
    }

    // ---- per-nonzero records (coalesced index/value loads) + linear term
    __syncwarp();
    double lin = 0.0;
    for (int u = gl; u < z; u += G) {
      NnzMeta m;
      if (u < zReal) {
        m.j = a.indices[rb + u];
        m.x = a.data[rb + u];
        double wj = a.w[m.j];
        const double xo = m.x;
        if constexpr (MODE == MODE_GRAD) {
          if (a.lazyInv) {
            // the shrink this feature has not received yet goes into x (ANOVA sees only p*x); the
            // gradient then comes out times the same factor and the lazy step divides it back
            const double2 iv = a.lazyInv[m.j];
            wj *= a.lazyCumWt * iv.y;
            m.x *= a.lazyCumPt * iv.x;
            a.lazyFlag[m.j] = 1;
          }
        }
        lin += wj * xo;
        m.acc = -1;
        if (MODE != MODE_PREDICT && a.hotSlot) {
          const int slot = a.hotSlot[m.j];
          if (slot != NIMFM_COLD) m.acc = slot * ASTR;
        }
      } else {
        m.j = (int32_t)(a.d + (u - zReal));
        m.x = 1.0;
        if constexpr (MODE == MODE_GRAD) {
          if (a.lazyInv) {
            m.x = a.lazyCumPt * a.lazyInv[m.j].x;
            a.lazyFlag[m.j] = 1;
          }
        }
        m.acc = (MODE != MODE_PREDICT) ? (a.nHot + (u - zReal)) * ASTR : -1;
      }
      sMeta[u] = m;
    }
    __syncwarp();

    // ---- forward: stream the P slice through registers, U nonzeros at a time (sgd.nim:146-173)
    double A[NO][DEGREE + 1];
#pragma unroll
    for (int o = 0; o < NO; ++o) {
      A[o][0] = 1.0;
#pragma unroll
      for (int t = 1; t <= DEGREE; ++t) A[o][t] = 0.0;
    }
    for (int c = 0; c < zmax; c += U) {
      double p[NO][U];
#pragma unroll
      for (int i = 0; i < U; ++i) {
        const bool ok = c + i < z;
        const int64_t j = ok ? (int64_t)sMeta[c + i].j : 0;
#pragma unroll
        for (int o = 0; o < NO; ++o) p[o][i] = ok ? __ldg(Pg + j * SB8 + o * KT) : 0.0;
      }
#pragma unroll
      for (int i = 0; i < U; ++i) {
        const double x = (c + i < z) ? sMeta[c + i].x : 0.0;
#pragma unroll
        for (int o = 0; o < NO; ++o) {
          const int M = DEGREE - o;
          const double t = p[o][i] * x;
          if (M == 2) {
            A[o][1] += t;
            A[o][2] += t * t;
          } else {
#pragma unroll
            for (int tt = DEGREE; tt >= 1; --tt)
              if (tt <= M) A[o][tt] += A[o][tt - 1] * t;
          }
        }
      }
    }
    double part = 0.0;
#pragma unroll
    for (int o = 0; o < NO; ++o) {
      const int M = DEGREE - o;
      if (M == 2) A[o][2] = (A[o][1] * A[o][1] - A[o][2]) / 2.0;
      part += A[o][M];
    }
    if (MODE == MODE_PREDICT && a.lams != nullptr) part *= a.lams[gl];
    double ysum = lin + part;
#pragma unroll
    for (int off = G >> 1; off > 0; off >>= 1) ysum += __shfl_xor_sync(0xffffffffu, ysum, off);
    const double yhat = bias + ysum;

    if (MODE == MODE_PREDICT) {
      if (active && gl == 0 && a.yOut) a.yOut[q] = yhat;
      continue;
    }
    if (MODE == MODE_STASH) {
      // forward half of the deterministic gradient (fm_cols.cu): what the derivative recurrence of sgd.nim:176-188
      // needs from this row -- coef and A[o][1 .. M_o-1] per component -- goes to the row's stash record
      if (active) {
        const double yi = a.y[r];
        const double dL = dev_dloss(a.loss, a.thr, yi, yhat);
        double *rec = a.stash + (size_t)q * a.stashStride;
        if (gl == 0) {
          if (a.yOut) a.yOut[q] = yhat;
          accLoss += dev_loss(a.loss, a.thr, yi, yhat);
          accB1 += dL / a.mb;
          accB2 += dL * dL;
          rec[0] = dL / a.mb;
        }
        int off = 1;
#pragma unroll
        for (int o = 0; o < NO; ++o) {
          const int M = DEGREE - o;
#pragma unroll
          for (int t = 1; t < DEGREE; ++t)
            if (t < M) {
              rec[off + gl] = A[o][t];
              off += KT;
            }
        }
      }
      continue;
    }

    // ---- loss derivative (loss.nim) and backward (sgd.nim:176-188 + minibatch_psgd.nim:73-88)
    double coef = 0.0;
    if (active) {
      if (a.yOut && gl == 0) a.yOut[q] = yhat;
      const double yi = a.y[r];
      const double dL = dev_dloss(a.loss, a.thr, yi, yhat);
      coef = (MODE == MODE_GRAD) ? dL / a.mb : dL;
      if (gl == 0) {
        accLoss += dev_loss(a.loss, a.thr, yi, yhat);
        accB1 += coef;
        accB2 += dL * dL;
      }
    }
    double *__restrict__ gPg = a.gP + gl;
    double *__restrict__ gNg = (MODE == MODE_ADAGRAD) ? a.dGnP + gl : nullptr;
    for (int c = 0; c < zmax; c += U) {
      double p[NO][U];
#pragma unroll
      for (int i = 0; i < U; ++i) {   // re-gather: these lines were read a moment ago (L1 / L2 hits)
        const bool ok = c + i < z;
        const int64_t j = ok ? (int64_t)sMeta[c + i].j : 0;
#pragma unroll
        for (int o = 0; o < NO; ++o) p[o][i] = ok ? __ldg(Pg + j * SB8 + o * KT) : 0.0;
      }
#pragma unroll
      for (int i = 0; i < U; ++i) {
        if (c + i < z) {
          const NnzMeta m = sMeta[c + i];
          double gr[NO];
#pragma unroll
          for (int o = 0; o < NO; ++o) {
            const int M = DEGREE - o;
            const double pv = p[o][i];
            double g;
            if (M == 2) {
              g = m.x * (A[o][1] - pv * m.x);
            } else {
              g = m.x;
#pragma unroll
              for (int tt = 1; tt < DEGREE; ++tt)
                if (tt < M) g = m.x * (A[o][tt] - pv * g);
            }
            gr[o] = coef * g;
          }
          if (m.acc >= 0) {   // hot column: lane-private shared accumulator element
            double *ac = sAcc + m.acc + gl;
#pragma unroll
            for (int o = 0; o < NO; ++o) ac[o * KT] += gr[o];
            if (MODE == MODE_ADAGRAD) {
              double *an = sAccN + m.acc + gl;
#pragma unroll
              for (int o = 0; o < NO; ++o) an[o * KT] += gr[o] * gr[o];
            }
            // linear-term gradient of a hot column: element SB8 of the slot is owned by the group's lane 0
            // (plain adds in nonzero order; a shared-memory FP64 atomicAdd is a CAS spin loop)
            if (gl == 0 && a.fitLinear && c + i < zReal) {
              const double gx = coef * m.x;
              sAcc[m.acc + SB8] += gx;
              if (MODE == MODE_ADAGRAD) sAccN[m.acc + SB8] += gx * gx;
            }
          } else {
            const int64_t eo = (int64_t)m.j * SB8;
#pragma unroll
            for (int o = 0; o < NO; ++o) atomicAdd(gPg + eo + o * KT, gr[o]);
            if (MODE == MODE_ADAGRAD) {
#pragma unroll
              for (int o = 0; o < NO; ++o) atomicAdd(gNg + eo + o * KT, gr[o] * gr[o]);
            }
          }
        }
      }
    }
    // ---- linear-term gradient of the cold real features: one lane per nonzero (hot columns: above)
    if (a.fitLinear) {
      for (int u = gl; u < zReal; u += G) {
        const NnzMeta m = sMeta[u];
        if (m.acc >= 0) continue;
        const double gx = coef * m.x;
        atomicAdd(a.gw + m.j, gx);
        if (MODE == MODE_ADAGRAD) atomicAdd(a.dGnw + m.j, gx * gx);
      }
    }
  }

  if constexpr (MODE == MODE_GRAD || MODE == MODE_ADAGRAD) {
    // ---- flush the hot-column accumulators ONCE PER BLOCK: the block's groups are summed in a fixed
    // order by one thread per element, then one RED per element (per-group flushes made every group
    // of a small minibatch hammer the same few hundred addresses: 180 us for 25 641 rows)
    __syncthreads();
    const int nGroupsInBlock = warpsPerBlock * GPW;
    const int perAcc = nHotTot * ASTR;
    const unsigned char *accBase = smem_raw + (size_t)CH * sizeof(NnzMeta);
    for (int e = threadIdx.x; e < perAcc * NACC; e += blockDim.x) {
      double v = 0.0;
      for (int g = 0; g < nGroupsInBlock; ++g)
        v += reinterpret_cast<const double *>(accBase + (size_t)g * perGroup)[e];
      if (v == 0.0) continue;
      const int which = e / perAcc, r = e - which * perAcc;
      const int slot = r / ASTR, c = r - slot * ASTR;
      const int64_t j = slot < a.nHot ? (int64_t)a.hotList[slot] : a.d + (slot - a.nHot);
      if (c < SB8) {
        atomicAdd((which ? a.dGnP : a.gP) + j * SB8 + c, v);
      } else if (a.fitLinear && j < a.d) {
        atomicAdd((which ? a.dGnw : a.gw) + j, v);
      }
    }
  }
  if constexpr (MODE != MODE_PREDICT) {
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

// The row kernels of one mode for (degree, explicit lower orders, k): the streaming instance (degree 2 / 3 with k in
// {8, 16, 32}, else null) and the generic runtime-k kernel (degree 2..6, else null).
struct RowKernels {
  RowKernel stream, generic;
};

template <int DEGREE, bool EXPLICIT, int MODE>
RowKernels row_kernels_of(int k) {
  RowKernels r{nullptr, fm_rows_kernel<DEGREE, EXPLICIT, MODE, 0>};
  if constexpr (DEGREE <= 3) {
    switch (k) {
      case 8: r.stream = fm_rows_stream_kernel<DEGREE, EXPLICIT, MODE, 8>; break;
      case 16: r.stream = fm_rows_stream_kernel<DEGREE, EXPLICIT, MODE, 16>; break;
      case 32: r.stream = fm_rows_stream_kernel<DEGREE, EXPLICIT, MODE, 32>; break;
    }
  }
  return r;
}

template <int MODE>
RowKernels row_kernels(int degree, bool explicitLower, int k) {
  switch (degree) {
    case 2: return row_kernels_of<2, false, MODE>(k);
    case 3: return explicitLower ? row_kernels_of<3, true, MODE>(k) : row_kernels_of<3, false, MODE>(k);
    case 4: return explicitLower ? row_kernels_of<4, true, MODE>(k) : row_kernels_of<4, false, MODE>(k);
    case 5: return explicitLower ? row_kernels_of<5, true, MODE>(k) : row_kernels_of<5, false, MODE>(k);
    case 6: return explicitLower ? row_kernels_of<6, true, MODE>(k) : row_kernels_of<6, false, MODE>(k);
    default: return {nullptr, nullptr};
  }
}

// Each mode is instantiated in its own translation unit, so the kernel families compile in parallel:
// fm_rows_predict.cu, fm_rows_grad.cu, fm_rows_adagrad.cu and fm_cols.cu (MODE_STASH).
extern template RowKernels row_kernels<MODE_PREDICT>(int, bool, int);
extern template RowKernels row_kernels<MODE_GRAD>(int, bool, int);
extern template RowKernels row_kernels<MODE_ADAGRAD>(int, bool, int);
extern template RowKernels row_kernels<MODE_STASH>(int, bool, int);
