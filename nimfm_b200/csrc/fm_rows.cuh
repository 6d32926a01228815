// fm_rows.cuh -- the row-parallel FM/HOFM kernel family (SURVEY K1, K2, K4).
//
// One GROUP of G lanes (G = 8, 16 or 32, a power of two >= min(k, 32)) owns one CSR row; lane <->
// component s.  Per row:
//   1. the row's (index, value) pairs are read with coalesced loads into shared memory, dummy
//      features (d+a, 1.0) appended (dataset.nim:182-189);
//   2. the row's P slice -- nnz x (nOrders*k) doubles, one contiguous nOrders*k*8-byte block per
//      nonzero thanks to the P[j][o][s] device layout -- is staged in shared memory with cp.async
//      (16 B per lane, all copies of the row in flight at once);
//   3. forward: the degree-m ANOVA dynamic program (sgd.nim:146-173; degree 2 uses the closed form
//      (A1^2-A2)/2, :160-170) runs out of shared memory for all orders, the linear term is gathered,
//      the group is reduced with warp shuffles, loss / dloss are evaluated (loss.nim);
//   4. backward (MODE_GRAD / MODE_ADAGRAD): the derivative recurrence (sgd.nim:176-188) re-reads the
//      staged slice (no second gather) and scatters coef*dA with FP64 RED atomics
//      (minibatch_psgd.nim:77-88 / adagrad.nim:113-134);
//   4'. MODE_STASH (the deterministic gradient, fm_cols.cu): no backward pass; each component chunk's
//      A[o][1 .. M_o-1] and the row's coef go to the row's stash record, which the column kernels read.
// Hot features: columns present in a large fraction of the rows (dense numeric columns, dummy features
// of fitLower=augment) would serialise ~nRows RED operations on the same few L2 addresses.  The dataset
// carries a byte table hotSlot[j] (built from a row sample at upload); gradients of hot features are
// accumulated in per-group shared-memory accumulators (each element owned by exactly one lane, so no
// shared atomics or barriers) and flushed with one RED per element when the kernel ends.
// Rows longer than the staging capacity CH are processed in chunks (the backward pass re-stages).
// k > G is handled by looping component chunks (the forward is recomputed per chunk in backward).
#pragma once
#include "common.cuh"

enum { MODE_PREDICT = 0, MODE_GRAD = 1, MODE_ADAGRAD = 2, MODE_STASH = 3 };

struct RowArgs {
  // dataset (CSR)
  const double *data;
  const int32_t *indices;
  const int64_t *indptr;
  const double *y;
  int64_t n;
  // rows to process: rowIdx[q] or (rowBegin + q) mod n, q < nRows
  int64_t rowBegin, nRows;
  const int32_t *rowIdx;
  // model
  int k, nAug;
  int64_t d;
  const double *P, *w, *b, *lams;
  int fitLinear, fitIntercept;
  // outputs
  double *yOut;       // nullable, yOut[q]
  double *gP, *gw;    // MODE_GRAD: gradient buffers; MODE_ADAGRAD: delta g_sum buffers
  double *partials;   // [nWarps][4]: loss, sum coef (gb) | sum dL, viol | sum dL^2, 0
  int loss;
  double thr, mb;     // coef = dloss / mb (minibatch_psgd.nim:73)
  // AdaGrad only (adagrad.nim:87-134)
  const double *gsP, *gnP, *gsw, *gnw, *adaScal;
  double *dGnP, *dGnw;
  double *touched;    // per-feature touch marker (part of the all-reduced delta block)
  double eta0, tIt, alpha0, alpha, beta;   // tIt = float(it-1)
  int first;                               // it == 1: no refresh
  // hot-feature accumulators (nullable table: no data-driven hot features)
  const uint8_t *hotSlot;   // [d], 255 = cold
  const int32_t *hotList;   // [nHot] feature id of each slot
  int nHot;
  // lazy L2 shrink of MBPSGD (fm_api.cu, "lazy" epoch): feature j was last brought up to date at inner
  // step l(j); its effective parameters are the stored ones times cum[t] / cum[l(j)], with
  // lazyInv[j] = {1 / cumP[l(j)], 1 / cumW[l(j)]}
  const double2 *lazyInv;           // nullptr: parameters are current (every other caller)
  double lazyCumPt, lazyCumWt;      // cum[t] of the current inner step
  uint8_t *lazyFlag;                // [d+nAug] set for every feature this minibatch touches
  // MODE_STASH (deterministic gradient, fm_cols.cu): per row [coef | A[o][1..M_o-1][s] ...], stashStride doubles
  double *stash;
  int stashStride;
  // geometry
  int G, CH;
};

typedef void (*RowKernel)(const RowArgs);

// one launch of a row kernel, as plan_rows (fm_api.cu) chooses it
struct RowPlan {
  RowKernel kern;
  bool stream;   // kern is the register-streaming instance (fm_rows_stream.cuh), else the generic kernel
  int G, CH, block, grid;
  size_t smem;
  int64_t nWarps;
};

// fm_linear.cu: the plan of the degree-1 (nOrders = 0) row kernel, which plan_rows returns for a model without P
int nimfm_fm_linear_plan(nimfm_ctx *ctx, const nimfm_dataset *X, int64_t nRows, int mode, RowPlan *pl);

// where the deterministic route's outputs go (nimfm_fm_det_pass)
struct FmDetTargets {
  double *gP = nullptr, *gw = nullptr;     // gradient sums (the model's gradient, g_sum or its delta block)
  double *gnP = nullptr, *gnw = nullptr;   // AdaGrad: sums of squared gradients; nullptr: plain gradient
  double *red4 = nullptr;                  // (loss, sum coef, sum dL^2, -)
  double *yhat = nullptr;   // [nRows] scratch: when set, red4 is summed from the rows' yhat by dloss_coef_kernel, in an
                            // order that does not depend on which forward kernel ran (AdaGrad: red4 moves the intercept)
};

#define NIMFM_COLD 255
#define NIMFM_MAX_HOT 16

// bytes of shared memory one row group needs (must match the carve-up in fm_rows_kernel)
__host__ __device__ inline size_t row_group_smem(int CH, int SB8, int nHotTot, int nAcc) {
  size_t b = ((size_t)CH * SB8 + CH + (size_t)nHotTot * (SB8 + 1) * nAcc) * 8 + (size_t)CH * 4 + (size_t)CH;
  return (b + 15) & ~(size_t)15;
}

template <int DEGREE, bool EXPLICIT>
struct RowCfg {
  static constexpr int NO = (EXPLICIT && DEGREE > 2) ? DEGREE - 1 : 1;
};

// KT > 0 fixes nComponents at compile time (KT in {8,16,32}: one lane per component, all index
// arithmetic constant-folded); KT == 0 is the generic runtime-k kernel.
template <int DEGREE, bool EXPLICIT, int MODE, int KT>
__global__ void __launch_bounds__(256, 1) fm_rows_kernel(const RowArgs a) {
  constexpr int NO = RowCfg<DEGREE, EXPLICIT>::NO;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x & 31;
  const int warpInBlock = threadIdx.x >> 5;
  const int G = KT ? (KT < 8 ? 8 : KT) : a.G;
  const int CH = a.CH;
  const int k = KT ? KT : a.k;
  const int gpw = 32 / G;
  const int gl = lane & (G - 1);
  const int gidInWarp = lane / G;
  const int SB8 = NO * k;  // doubles per feature slice
  constexpr int NACC = (MODE == MODE_ADAGRAD) ? 2 : 1;
  const int nHotTot = (MODE == MODE_PREDICT || MODE == MODE_STASH) ? 0 : a.nHot + a.nAug;
  const int ASTR = SB8 + 1;  // accumulator stride per slot: SB8 P-gradients + 1 w-gradient
  const size_t perGroup = row_group_smem(CH, SB8, nHotTot, NACC);
  unsigned char *base = smem_raw + (size_t)(warpInBlock * gpw + gidInWarp) * perGroup;
  double *sP = reinterpret_cast<double *>(base);
  double *sVal = sP + (size_t)CH * SB8;
  double *sAcc = sVal + CH;                               // [nHotTot][ASTR] gradient sums
  double *sAccN = sAcc + (size_t)nHotTot * ASTR;          // AdaGrad: squared-gradient sums
  int *sIdx = reinterpret_cast<int *>(sAcc + (size_t)nHotTot * ASTR * NACC);
  unsigned char *sSlot = reinterpret_cast<unsigned char *>(sIdx + CH);
  for (int e = gl; e < nHotTot * ASTR * NACC; e += G) sAcc[e] = 0.0;
  __syncwarp();

  const int warpsPerBlock = blockDim.x >> 5;
  const int64_t warpGlobal = (int64_t)blockIdx.x * warpsPerBlock + warpInBlock;
  const int64_t nWarps = (int64_t)gridDim.x * warpsPerBlock;
  const int64_t tiles = (a.nRows + gpw - 1) / gpw;
  const int NS = (k + G - 1) / G;

  double accLoss = 0.0, accB1 = 0.0, accB2 = 0.0, accViol = 0.0;

  // AdaGrad: the intercept every row of this batch sees (adagrad.nim:101-105)
  double bias = a.b[0];
  if (MODE == MODE_ADAGRAD) {
    if (!a.first && a.fitIntercept) {
      double den = sqrt(a.adaScal[1]) + a.eta0 * a.tIt * a.alpha0;
      bias = -a.eta0 * a.adaScal[0] / den;
    }
  }

  for (int64_t tile = warpGlobal; tile < tiles; tile += nWarps) {
    const int64_t q = tile * gpw + gidInWarp;
    const bool active = q < a.nRows;
    int64_t r = 0;
    if (active) r = a.rowIdx ? (int64_t)a.rowIdx[q] : (a.rowBegin + q) % a.n;
    const int64_t rb = active ? a.indptr[r] : 0;
    const int zReal = active ? (int)(a.indptr[r + 1] - rb) : 0;
    const int z = active ? zReal + a.nAug : 0;
    int zmax = z;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) zmax = max(zmax, __shfl_xor_sync(0xffffffffu, zmax, off));
    const int nChunks = (zmax + CH - 1) / CH;

    // ---- stage chunk c of every group of this warp (warp-uniform call)
    auto stage = [&](int c, bool withLinear, double &lin) {
      const int c0 = c * CH;
      int cnt = z - c0;
      cnt = cnt < 0 ? 0 : (cnt > CH ? CH : cnt);
      __syncwarp();
      for (int u = gl; u < cnt; u += G) {
        const int pos = c0 + u;
        int j;
        double x;
        if (pos < zReal) {
          j = a.indices[rb + pos];
          x = a.data[rb + pos];
        } else {
          j = (int)(a.d + (pos - zReal));
          x = 1.0;
        }
        sIdx[u] = j;
        sVal[u] = x;
        if (MODE != MODE_PREDICT && MODE != MODE_STASH)
          sSlot[u] = pos >= zReal ? (unsigned char)(a.nHot + (pos - zReal))
                                  : (a.hotSlot ? a.hotSlot[j] : (unsigned char)NIMFM_COLD);
        if (withLinear && pos < zReal) lin += a.w[j] * x;
      }
      __syncwarp();
      // (AdaGrad: P was refreshed from (g_sum, g_norm, t) by adagrad_refresh_kernel before this launch)
      if ((SB8 & 1) == 0) {
        const int units = SB8 >> 1;
        const int total = cnt * units;
        if ((units & (units - 1)) == 0) {
          const int sh = __ffs(units) - 1;
          for (int u = gl; u < total; u += G) {
            const int qq = u >> sh, off = (u & (units - 1)) << 1;
            cp_async16(sP + (size_t)qq * SB8 + off, a.P + (int64_t)sIdx[qq] * SB8 + off);
          }
        } else {
          for (int u = gl; u < total; u += G) {
            const int qq = u / units, off = (u - qq * units) << 1;
            cp_async16(sP + (size_t)qq * SB8 + off, a.P + (int64_t)sIdx[qq] * SB8 + off);
          }
        }
      } else {
        const int total = cnt * SB8;
        for (int u = gl; u < total; u += G) {
          const int qq = u / SB8, off = u - qq * SB8;
          cp_async8(sP + (size_t)qq * SB8 + off, a.P + (int64_t)sIdx[qq] * SB8 + off);
        }
      }
      cp_async_wait_all();
      __syncwarp();
    };

    // ---- forward over one staged chunk for component s (lane-private DP state A)
    auto fwd_chunk = [&](int c, int s, double (&A)[NO][DEGREE + 1]) {
      const int c0 = c * CH;
      int cnt = z - c0;
      cnt = cnt < 0 ? 0 : (cnt > CH ? CH : cnt);
      if (s >= k) cnt = 0;
      for (int u = 0; u < cnt; ++u) {
        const double x = sVal[u];
        const double *ps = sP + (size_t)u * SB8 + s;
#pragma unroll
        for (int o = 0; o < NO; ++o) {
          const int M = DEGREE - o;
          const double t = ps[o * k] * x;
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
    };

    auto fwd_all = [&](int sc, double (&A)[NO][DEGREE + 1], bool withLinear, double &lin) -> double {
      const int s = sc * G + gl;
#pragma unroll
      for (int o = 0; o < NO; ++o) {
        A[o][0] = 1.0;
#pragma unroll
        for (int tt = 1; tt <= DEGREE; ++tt) A[o][tt] = 0.0;
      }
      for (int c = 0; c < nChunks; ++c) {
        if (nChunks > 1) {
          stage(c, withLinear, lin);
        }
        fwd_chunk(c, s, A);
      }
      double acc = 0.0;
#pragma unroll
      for (int o = 0; o < NO; ++o) {
        const int M = DEGREE - o;
        if (M == 2) A[o][2] = (A[o][1] * A[o][1] - A[o][2]) / 2.0;
        acc += A[o][M];
      }
      if (s >= k) acc = 0.0;
      if (MODE == MODE_PREDICT && a.lams != nullptr && s < k) acc *= a.lams[s];
      return acc;
    };

    double lin = 0.0;
    double A[NO][DEGREE + 1];
    if (nChunks == 1) stage(0, true, lin);
    double part = 0.0;
    for (int sc = 0; sc < NS; ++sc) {
      part += fwd_all(sc, A, sc == 0, lin);
      if (MODE == MODE_STASH) {
        // the row's stash record (fm_cols.cu) takes A[o][1 .. M_o-1] of this component chunk, laid out like the
        // streaming kernel's: [coef | A[o][t][s] for o, t = 1 .. M_o-1, s < k]
        const int s = sc * G + gl;
        if (active && s < k) {
          double *rec = a.stash + (size_t)q * a.stashStride + 1 + s;
          int off = 0;
#pragma unroll
          for (int o = 0; o < NO; ++o) {
            const int M = DEGREE - o;
#pragma unroll
            for (int tt = 1; tt < DEGREE; ++tt)
              if (tt < M) {
                rec[off] = A[o][tt];
                off += k;
              }
          }
        }
      }
    }
    // (for nChunks == 1 the staged slice stays resident for the backward pass)
    const double yhat = bias + group_sum(lin + part, G);

    double dL = 0.0, coef = 0.0;
    if (active) {
      if (a.yOut && gl == 0) a.yOut[q] = yhat;
      if (MODE != MODE_PREDICT) {
        const double yi = a.y[r];
        dL = dev_dloss(a.loss, a.thr, yi, yhat);
        coef = (MODE == MODE_GRAD || MODE == MODE_STASH) ? dL / a.mb : dL;
        if (gl == 0) {
          accLoss += dev_loss(a.loss, a.thr, yi, yhat);
          accB1 += coef;
          accB2 += dL * dL;
          if (MODE == MODE_STASH) a.stash[(size_t)q * a.stashStride] = coef;
        }
      }
    }

    if (MODE != MODE_PREDICT && MODE != MODE_STASH) {
      for (int sc = NS - 1; sc >= 0; --sc) {
        const int s = sc * G + gl;
        if (sc != NS - 1) {
          double dummyLin = 0.0;
          (void)fwd_all(sc, A, false, dummyLin);  // recompute this component chunk's DP state
        }
        for (int c = 0; c < nChunks; ++c) {
          if (nChunks > 1) {
            double dummyLin = 0.0;
            stage(c, false, dummyLin);
          }
          const int c0 = c * CH;
          int cnt = z - c0;
          cnt = cnt < 0 ? 0 : (cnt > CH ? CH : cnt);
          if (s < k) {
            for (int u = 0; u < cnt; ++u) {
              const double x = sVal[u];
              const int64_t e0 = (int64_t)sIdx[u] * SB8 + s;
              const double *ps = sP + (size_t)u * SB8 + s;
              const int slot = sSlot[u];
              if (slot != NIMFM_COLD && sc == 0 && gl == 0 && a.fitLinear && sIdx[u] < a.d) {
                const double gx = coef * x;               // w-gradient of a hot feature: owned by lane 0
                sAcc[slot * ASTR + SB8] += gx;
                if (MODE == MODE_ADAGRAD) sAccN[slot * ASTR + SB8] += gx * gx;
              }
#pragma unroll
              for (int o = 0; o < NO; ++o) {
                const int M = DEGREE - o;
                const double p = ps[o * k];
                double g;
                if (M == 2) {
                  g = x * (A[o][1] - p * x);
                } else {
                  g = x;
#pragma unroll
                  for (int tt = 1; tt < DEGREE; ++tt)
                    if (tt < M) g = x * (A[o][tt] - p * g);
                }
                const double gr = coef * g;
                if (slot != NIMFM_COLD) {                  // element (slot, o, s) is private to this lane
                  sAcc[slot * ASTR + o * k + s] += gr;
                  if (MODE == MODE_ADAGRAD) sAccN[slot * ASTR + o * k + s] += gr * gr;
                } else {
                  atomicAdd(a.gP + e0 + o * k, gr);
                  if (MODE == MODE_ADAGRAD) atomicAdd(a.dGnP + e0 + o * k, gr * gr);
                }
              }
            }
          }
          if (sc == 0) {
            // linear-term gradient (real features only) and AdaGrad touched flags
            for (int u = gl; u < cnt; u += G) {
              const int j = sIdx[u];
              if (a.fitLinear && j < a.d && sSlot[u] == NIMFM_COLD) {
                const double gx = coef * sVal[u];
                atomicAdd(a.gw + j, gx);
                if (MODE == MODE_ADAGRAD) atomicAdd(a.dGnw + j, gx * gx);
              }
            }
          }
        }
      }
    }
    __syncwarp();
  }

  if (MODE != MODE_PREDICT && MODE != MODE_STASH && nHotTot > 0) {
    // flush the hot-feature accumulators: every lane writes the elements it owns
    __syncwarp();
    for (int slot = 0; slot < nHotTot; ++slot) {
      const int64_t j = slot < a.nHot ? (int64_t)a.hotList[slot] : a.d + (slot - a.nHot);
      for (int s = gl; s < k; s += G) {
#pragma unroll
        for (int o = 0; o < NO; ++o) {
          const double v = sAcc[slot * ASTR + o * k + s];
          if (v != 0.0) atomicAdd(a.gP + j * SB8 + o * k + s, v);
          if (MODE == MODE_ADAGRAD) {
            const double v2 = sAccN[slot * ASTR + o * k + s];
            if (v2 != 0.0) atomicAdd(a.dGnP + j * SB8 + o * k + s, v2);
          }
        }
      }
      if (gl == 0 && a.fitLinear && j < a.d) {
        const double v = sAcc[slot * ASTR + SB8];
        if (v != 0.0) atomicAdd(a.gw + j, v);
        if (MODE == MODE_ADAGRAD) {
          const double v2 = sAccN[slot * ASTR + SB8];
          if (v2 != 0.0) atomicAdd(a.dGnw + j, v2);
        }
      }
    }
  }

  if (MODE != MODE_PREDICT) {
    accLoss = warp_sum(accLoss);
    accB1 = warp_sum(accB1);
    accB2 = warp_sum(accB2);
    accViol = warp_sum(accViol);
    if (lane == 0) {
      a.partials[warpGlobal * 4 + 0] = accLoss;
      a.partials[warpGlobal * 4 + 1] = accB1;
      a.partials[warpGlobal * 4 + 2] = accB2;
      a.partials[warpGlobal * 4 + 3] = accViol;
    }
  }
}
