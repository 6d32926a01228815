// fm_cols.cu -- the DETERMINISTIC predict+grad route (NIMFM_DETERMINISTIC=1): no atomics anywhere.
//
// The reference accumulates a minibatch's gradient sample by sample (minibatch_psgd.nim:77-85), so its sums have
// ONE order; the default device route (fm_rows_stream.cuh) scatters with FP64 REDs, whose order changes from
// run to run (~1e-16 relative noise).  This route fixes the order instead:
//   pass 1  the row kernel in MODE_STASH: forward + loss derivative; each row leaves a stash record
//           [coef | A[o][1 .. M_o-1][s]] -- everything the derivative recurrence of sgd.nim:176-188 needs from the row;
//   pass 2  a COLUMN kernel over the CSC twin of the dataset (stable transpose: rows ascending inside a column):
//           for feature j, the entries of column j inside the row range are walked in row order, lane <-> component,
//           the parameter row P[j][o][s] sits in registers, every entry contributes coef_i * dA_i(j, o, s) to a register
//           accumulator, and the sum is written with ONE plain store per gradient element.  Long columns are cut
//           into segments of SEG entries whose partial sums a second kernel adds in segment order.
// Every gradient element is therefore a sum in ascending row order over fixed segments: bit-identical from run
// to run and independent of the grid.  Traffic per nonzero: 12 B of CSC + the row's stash record (M_o-1 values per
// component: 128 B for C3, 768 B for C4) instead of a re-gather of P and a RED; no read-for-ownership of cold
// gradient lines.
// Two forms of each pass, which read and write the same stash record (stride 1 + k * sum_o (M_o - 1), padded to an
// even number of doubles) and therefore combine either way:
//   tuned    the streaming row kernel (fm_rows_stream.cuh) and fm_cols_grad_kernel<D, E, KT>: degree 2 / 3,
//            k in {8,16,32}, rows of at most 512 nonzeros incl. dummy features;
//   generic  the runtime-k row kernel (fm_rows.cuh, chunked long rows and component chunks) and
//            fm_cols_grad_generic_kernel<D, E>: degree 2 .. 6, every k, rows of any length.
// The tuned pair runs where the streaming forward runs; every other shape, and NIMFM_ROW_KERNEL=generic, takes the
// generic pair.  Both need a contiguous row range without wrap-around (no row list).
#include <stdlib.h>

#include <algorithm>

#include "dense_kernels.cuh"
#include "fm_rows_stream.cuh"

// the stash forwards: the streaming instances and the generic runtime-k kernel (every degree, every k, any row length)
template RowKernels row_kernels<MODE_STASH>(int, bool, int);

namespace {

constexpr int SEG = 512;   // entries per column segment

struct ColArgs {
  const double *cdata;      // CSC values
  const int32_t *crow;      // CSC row ids (ascending inside a column)
  const int32_t *taskCol;   // [nTasks] feature id (>= d: dummy feature d + a)
  const int64_t *taskBeg;   // [nTasks] first entry of the segment (dummy features: first row)
  const int32_t *taskLen;   // [nTasks]
  const int32_t *taskSlot;  // [nTasks] partial-sum slot, -1: the segment is the whole column
  int64_t nTasks;
  int64_t d, rowBegin, rowEnd;
  const double *P;
  const double *stash;
  int stashStride;
  double *gP, *gw;
  double *partial;          // [nSlots][SB8 + 1]; AdaGrad forms: [nSlots][2 (SB8 + 1)], sums then squares
  int fitLinear;
  int k, KT;                // fm_cols_grad_generic_kernel only: nComponents and the lane-group width
  double *gnP, *gnw;        // AdaGrad forms: where the squared gradients go (g_norm or its delta block)
};

// first position in [lo, hi) whose row id is >= r
__device__ __forceinline__ int64_t lower_bound_row(const int32_t *rows, int64_t lo, int64_t hi, int64_t r) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((int64_t)rows[mid] < r) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// ADA (AdaGrad, adagrad.nim:113-124): every entry's gradient g = coef * dA is rounded on its own, as the RED route adds
// it, and the kernel also sums g * g into gnP / gnw.  A CSR row holds a feature once, so an entry is the sample's whole
// gradient element and its square is the reference's.  The ADA instances ask for two resident blocks per SM: left to
// its default, ptxas holds <3, false, KT, true> to 64 registers and spills; the gradient instances keep no minimum.
template <int DEGREE, bool EXPLICIT, int KT, bool ADA = false>
__global__ void __launch_bounds__(256, ADA ? 2 : 0) fm_cols_grad_kernel(const ColArgs a) {
  constexpr int NO = RowCfg<DEGREE, EXPLICIT>::NO;
  constexpr int G = KT, GPW = 32 / G, SB8 = NO * KT, U = 4;
  const int lane = threadIdx.x & 31, gl = lane & (G - 1), gid = lane / G;
  const int64_t group = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
  const int64_t nGroups = (int64_t)gridDim.x * blockDim.x / G;
  (void)gid;
  (void)GPW;
  for (int64_t t = group; t < a.nTasks; t += nGroups) {
    const int64_t j = a.taskCol[t];
    const bool dummy = j >= a.d;
    int64_t eb = a.taskBeg[t], ee = eb + a.taskLen[t];
    if (!dummy) {   // clip the segment to the row range (rows ascend inside a column)
      if ((int64_t)a.crow[eb] < a.rowBegin) eb = lower_bound_row(a.crow, eb, ee, a.rowBegin);
      if (eb < ee && (int64_t)a.crow[ee - 1] >= a.rowEnd) ee = lower_bound_row(a.crow, eb, ee, a.rowEnd);
    } else {
      eb = eb < a.rowBegin ? a.rowBegin : eb;
      ee = ee > a.rowEnd ? a.rowEnd : ee;
    }
    double p[NO], acc[NO], accW = 0.0, accN[NO], accWN = 0.0;
#pragma unroll
    for (int o = 0; o < NO; ++o) {
      p[o] = a.P[j * SB8 + o * KT + gl];
      acc[o] = 0.0;
      accN[o] = 0.0;
    }
    // software pipeline: the row ids / values of batch b+1 are fetched while batch b's stash records are in flight,
    // so a batch costs ONE dependent memory latency (stash gather) instead of two (ncu on the unpipelined form:
    // long_scoreboard 21.6 warps per issue, DRAM at 38 % of peak)
    int64_t rowN[U];
    double xN[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t e = eb + u;
      const bool ok = e < ee;
      rowN[u] = ok ? (dummy ? e : (int64_t)a.crow[e]) : a.rowBegin;
      xN[u] = ok ? (dummy ? 1.0 : a.cdata[e]) : 0.0;
    }
    for (int64_t e0 = eb; e0 < ee; e0 += U) {
      double x[U], coef[U], av[U][NO][DEGREE];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const bool ok = e0 + u < ee;
        x[u] = xN[u];
        const double *rec = a.stash + (size_t)(rowN[u] - a.rowBegin) * a.stashStride;
        coef[u] = ok ? rec[0] : 0.0;
        int off = 1;
#pragma unroll
        for (int o = 0; o < NO; ++o) {
          const int M = DEGREE - o;
#pragma unroll
          for (int tt = 1; tt < DEGREE; ++tt)
            if (tt < M) {
              av[u][o][tt] = ok ? rec[off + gl] : 0.0;
              off += KT;
            }
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {   // next batch's entries
        const int64_t e = e0 + U + u;
        const bool ok = e < ee;
        rowN[u] = ok ? (dummy ? e : (int64_t)a.crow[e]) : a.rowBegin;
        xN[u] = ok ? (dummy ? 1.0 : a.cdata[e]) : 0.0;
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {   // entries in ascending row order: the sum has one order
#pragma unroll
        for (int o = 0; o < NO; ++o) {
          const int M = DEGREE - o;
          double g;
          if (M == 2) {
            g = x[u] * (av[u][o][1] - p[o] * x[u]);
          } else {
            g = x[u];
#pragma unroll
            for (int tt = 1; tt < DEGREE; ++tt)
              if (tt < M) g = x[u] * (av[u][o][tt] - p[o] * g);
          }
          if (ADA) {
            const double gr = __dmul_rn(coef[u], g);
            acc[o] += gr;
            accN[o] += __dmul_rn(gr, gr);
          } else {
            acc[o] += coef[u] * g;
          }
        }
        if (ADA) {
          const double gx = __dmul_rn(coef[u], x[u]);
          accW += gx;
          accWN += __dmul_rn(gx, gx);
        } else {
          accW += coef[u] * x[u];
        }
      }
    }
    const int slot = a.taskSlot[t];
    if (slot < 0) {
#pragma unroll
      for (int o = 0; o < NO; ++o) {
        a.gP[j * SB8 + o * KT + gl] += acc[o];
        if (ADA) a.gnP[j * SB8 + o * KT + gl] += accN[o];
      }
      if (gl == 0 && !dummy && a.fitLinear) {
        a.gw[j] += accW;
        if (ADA) a.gnw[j] += accWN;
      }
    } else {
      double *ps = a.partial + (size_t)slot * (ADA ? 2 : 1) * (SB8 + 1);
#pragma unroll
      for (int o = 0; o < NO; ++o) {
        ps[o * KT + gl] = acc[o];
        if (ADA) ps[SB8 + 1 + o * KT + gl] = accN[o];
      }
      if (gl == 0) {
        ps[SB8] = accW;
        if (ADA) ps[2 * SB8 + 1] = accWN;
      }
    }
  }
}

// fm_cols_grad_kernel with nComponents at run time (every degree, every k): a group of KT lanes (KT in {4,8,16,32},
// lane_group_kt) maps lane <-> component s = sc*KT + lane of component chunk sc, and a task walks its entries once per
// chunk; lanes past k idle.  Per entry the arithmetic is fm_cols_grad_kernel's expression sequence in the same
// ascending row order, so where both kernels run they produce the same bits.  ADA: as in fm_cols_grad_kernel; those
// instances are held to one 256-thread block per SM by their launch bounds, for room for the square accumulators.
template <int DEGREE, bool EXPLICIT, bool ADA = false>
__global__ void __launch_bounds__(256, ADA ? 1 : 2) fm_cols_grad_generic_kernel(const ColArgs a) {
  constexpr int NO = RowCfg<DEGREE, EXPLICIT>::NO;
  constexpr int NV = NO * (2 * DEGREE - NO - 1) / 2;   // stash values per component: sum over o of M_o - 1
  constexpr int U = NV <= 6 ? 4 : 2;                   // entries per batch (register budget of av below)
  const int k = a.k, KT = a.KT, SB8 = NO * k;
  const int gl = (threadIdx.x & 31) & (KT - 1);
  const int64_t group = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / KT;
  const int64_t nGroups = (int64_t)gridDim.x * blockDim.x / KT;
  const int NC = (k + KT - 1) / KT;
  for (int64_t t = group; t < a.nTasks; t += nGroups) {
    const int64_t j = a.taskCol[t];
    const bool dummy = j >= a.d;
    int64_t eb = a.taskBeg[t], ee = eb + a.taskLen[t];
    if (!dummy) {   // clip the segment to the row range (rows ascend inside a column)
      if ((int64_t)a.crow[eb] < a.rowBegin) eb = lower_bound_row(a.crow, eb, ee, a.rowBegin);
      if (eb < ee && (int64_t)a.crow[ee - 1] >= a.rowEnd) ee = lower_bound_row(a.crow, eb, ee, a.rowEnd);
    } else {
      eb = eb < a.rowBegin ? a.rowBegin : eb;
      ee = ee > a.rowEnd ? a.rowEnd : ee;
    }
    const int slot = a.taskSlot[t];
    for (int sc = 0; sc < NC; ++sc) {
      const int s = sc * KT + gl;
      if (s >= k) break;
      double p[NO], acc[NO], accW = 0.0, accN[NO], accWN = 0.0;
#pragma unroll
      for (int o = 0; o < NO; ++o) {
        p[o] = a.P[j * SB8 + o * k + s];
        acc[o] = 0.0;
        accN[o] = 0.0;
      }
      // the same software pipeline as fm_cols_grad_kernel: batch b+1's row ids / values load under batch b's records
      int64_t rowN[U];
      double xN[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t e = eb + u;
        const bool ok = e < ee;
        rowN[u] = ok ? (dummy ? e : (int64_t)a.crow[e]) : a.rowBegin;
        xN[u] = ok ? (dummy ? 1.0 : a.cdata[e]) : 0.0;
      }
      for (int64_t e0 = eb; e0 < ee; e0 += U) {
        double x[U], coef[U], av[U][NO][DEGREE];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const bool ok = e0 + u < ee;
          x[u] = xN[u];
          const double *rec = a.stash + (size_t)(rowN[u] - a.rowBegin) * a.stashStride;
          coef[u] = ok ? rec[0] : 0.0;
          int off = 1 + s;
#pragma unroll
          for (int o = 0; o < NO; ++o) {
            const int M = DEGREE - o;
#pragma unroll
            for (int tt = 1; tt < DEGREE; ++tt)
              if (tt < M) {
                av[u][o][tt] = ok ? rec[off] : 0.0;
                off += k;
              }
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {   // next batch's entries
          const int64_t e = e0 + U + u;
          const bool ok = e < ee;
          rowN[u] = ok ? (dummy ? e : (int64_t)a.crow[e]) : a.rowBegin;
          xN[u] = ok ? (dummy ? 1.0 : a.cdata[e]) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {   // entries in ascending row order: the sum has one order
#pragma unroll
          for (int o = 0; o < NO; ++o) {
            const int M = DEGREE - o;
            double g;
            if (M == 2) {
              g = x[u] * (av[u][o][1] - p[o] * x[u]);
            } else {
              g = x[u];
#pragma unroll
              for (int tt = 1; tt < DEGREE; ++tt)
                if (tt < M) g = x[u] * (av[u][o][tt] - p[o] * g);
            }
            if (ADA) {
              const double gr = __dmul_rn(coef[u], g);
              acc[o] += gr;
              accN[o] += __dmul_rn(gr, gr);
            } else {
              acc[o] += coef[u] * g;
            }
          }
          if (ADA) {
            const double gx = __dmul_rn(coef[u], x[u]);
            accW += gx;
            accWN += __dmul_rn(gx, gx);
          } else {
            accW += coef[u] * x[u];
          }
        }
      }
      if (slot < 0) {
#pragma unroll
        for (int o = 0; o < NO; ++o) {
          a.gP[j * SB8 + o * k + s] += acc[o];
          if (ADA) a.gnP[j * SB8 + o * k + s] += accN[o];
        }
        if (s == 0 && !dummy && a.fitLinear) {
          a.gw[j] += accW;
          if (ADA) a.gnw[j] += accWN;
        }
      } else {
        double *ps = a.partial + (size_t)slot * (ADA ? 2 : 1) * (SB8 + 1);
#pragma unroll
        for (int o = 0; o < NO; ++o) {
          ps[o * k + s] = acc[o];
          if (ADA) ps[SB8 + 1 + o * k + s] = accN[o];
        }
        if (s == 0) {
          ps[SB8] = accW;
          if (ADA) ps[2 * SB8 + 1] = accWN;
        }
      }
    }
  }
}

// The column pass of the degree-1 model (nOrders = 0, no P, no dummy features; the stash forward is fm_linear.cu's
// MODE_STASH): one thread per segment walks its entries in ascending row order and adds coef * x into one register,
// written with one plain store per column (or into the segment's partial slot, [w] / [w | w^2], for the combine
// kernels at SB8 = 0).  ADA: g = coef * x is rounded on its own and g * g is summed into gnw, as in the other forms.
template <bool ADA>
__global__ void __launch_bounds__(256) fm_cols_linear_kernel(const ColArgs a) {
  const int64_t nth = (int64_t)gridDim.x * blockDim.x;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < a.nTasks; t += nth) {
    const int64_t j = a.taskCol[t];
    int64_t eb = a.taskBeg[t], ee = eb + a.taskLen[t];
    if ((int64_t)a.crow[eb] < a.rowBegin) eb = lower_bound_row(a.crow, eb, ee, a.rowBegin);
    if (eb < ee && (int64_t)a.crow[ee - 1] >= a.rowEnd) ee = lower_bound_row(a.crow, eb, ee, a.rowEnd);
    double accW = 0.0, accWN = 0.0;
    for (int64_t e = eb; e < ee; ++e) {
      const double coef = a.stash[(size_t)((int64_t)a.crow[e] - a.rowBegin) * a.stashStride];
      if (ADA) {
        const double gx = __dmul_rn(coef, a.cdata[e]);
        accW += gx;
        accWN += __dmul_rn(gx, gx);
      } else {
        accW += coef * a.cdata[e];
      }
    }
    const int slot = a.taskSlot[t];
    if (slot < 0) {
      if (a.fitLinear) {
        a.gw[j] += accW;
        if (ADA) a.gnw[j] += accWN;
      }
    } else {
      double *ps = a.partial + (size_t)slot * (ADA ? 2 : 1);
      ps[0] = accW;
      if (ADA) ps[1] = accWN;
    }
  }
}

// columns cut into several segments: their partial sums are added in segment order
__global__ void fm_cols_combine_kernel(const int32_t *multiCol, const int32_t *multiFirst, const int32_t *multiCount,
                                       int64_t nMulti, const double *partial, int SB8, int64_t d, double *gP, double *gw,
                                       int fitLinear) {
  const int64_t c = blockIdx.x;
  if (c >= nMulti) return;
  const int64_t j = multiCol[c];
  for (int e = threadIdx.x; e <= SB8; e += blockDim.x) {
    double s = 0.0;
    const double *ps = partial + (size_t)multiFirst[c] * (SB8 + 1) + e;
    for (int q = 0; q < multiCount[c]; ++q) s += ps[(size_t)q * (SB8 + 1)];
    if (e < SB8) gP[j * SB8 + e] += s;
    else if (j < d && fitLinear) gw[j] += s;
  }
}

// the AdaGrad form: a slot holds the sums, then the sums of squares, [SB8 | w | SB8 | w]; the second half goes to gnP / gnw
__global__ void fm_cols_combine_ada_kernel(const int32_t *multiCol, const int32_t *multiFirst, const int32_t *multiCount,
                                           int64_t nMulti, const double *partial, int SB8, int64_t d, double *gP, double *gw,
                                           double *gnP, double *gnw, int fitLinear) {
  const int64_t c = blockIdx.x;
  if (c >= nMulti) return;
  const int64_t j = multiCol[c];
  const int S = 2 * (SB8 + 1);
  for (int e = threadIdx.x; e < S; e += blockDim.x) {
    double s = 0.0;
    const double *ps = partial + (size_t)multiFirst[c] * S + e;
    for (int q = 0; q < multiCount[c]; ++q) s += ps[(size_t)q * S];
    const int h = e <= SB8 ? e : e - (SB8 + 1);
    double *dP = e <= SB8 ? gP : gnP, *dW = e <= SB8 ? gw : gnw;
    if (h < SB8) dP[j * SB8 + h] += s;
    else if (j < d && fitLinear) dW[j] += s;
  }
}

typedef void (*ColKernel)(const ColArgs);
template <int DEGREE, bool EXPLICIT, bool ADA>
ColKernel pick_cols(int k) {
  switch (k) {
    case 8: return fm_cols_grad_kernel<DEGREE, EXPLICIT, 8, ADA>;
    case 16: return fm_cols_grad_kernel<DEGREE, EXPLICIT, 16, ADA>;
    case 32: return fm_cols_grad_kernel<DEGREE, EXPLICIT, 32, ADA>;
    default: return nullptr;
  }
}

template <bool ADA>
ColKernel pick_cols_generic(int degree, bool explicitLower) {
  switch (degree) {
    case 2: return fm_cols_grad_generic_kernel<2, false, ADA>;
    case 3: return explicitLower ? fm_cols_grad_generic_kernel<3, true, ADA> : fm_cols_grad_generic_kernel<3, false, ADA>;
    case 4: return explicitLower ? fm_cols_grad_generic_kernel<4, true, ADA> : fm_cols_grad_generic_kernel<4, false, ADA>;
    case 5: return explicitLower ? fm_cols_grad_generic_kernel<5, true, ADA> : fm_cols_grad_generic_kernel<5, false, ADA>;
    case 6: return explicitLower ? fm_cols_grad_generic_kernel<6, true, ADA> : fm_cols_grad_generic_kernel<6, false, ADA>;
    default: return nullptr;
  }
}

}  // namespace

void nimfm_det_twin_free(nimfm_ctx *ctx, nimfm_det_twin *t) {
  if (!t) return;
  nimfm_dataset_free(ctx, t->csc);
  cudaFree(t->taskCol); cudaFree(t->taskLen); cudaFree(t->taskSlot); cudaFree(t->taskBeg);
  cudaFree(t->multiCol); cudaFree(t->multiFirst); cudaFree(t->multiCount);
  delete t;
}

// The column twin of a CSR dataset and the segment list of its columns, built once per dataset (bookkeeping).
static int build_twin(nimfm_ctx *ctx, const nimfm_dataset *X, int nAug, nimfm_det_twin **out) {
  nimfm_det_twin *t = new nimfm_det_twin();
  struct Guard { nimfm_ctx *c; nimfm_det_twin *t; ~Guard() { if (t) nimfm_det_twin_free(c, t); } } guard{ctx, t};
  nimfm_dataset view = *X;      // a plain-CSR view of the same device arrays (a field dataset's fields play no part here)
  view.kind = NIMFM_DS_CSR;
  view.fields = nullptr;
  view.y = nullptr;
  view.detTwin = nullptr;
  int rc = nimfm_dataset_transpose(ctx, &view, &t->csc);
  if (rc) return rc;
  const int64_t d = X->d, n = X->n;
  std::vector<int64_t> ptr((size_t)d + 1);
  CK(cudaMemcpy(ptr.data(), t->csc->indptr, ((size_t)d + 1) * 8, cudaMemcpyDeviceToHost));
  std::vector<int32_t> col, len, slot, mcol, mfirst, mcount;
  std::vector<int64_t> beg;
  int64_t nSlots = 0;
  auto add_column = [&](int64_t j, int64_t b, int64_t e) {
    const int64_t L = e - b;
    if (L <= 0) return;
    const int64_t nseg = (L + SEG - 1) / SEG;
    if (nseg > 1) {
      mcol.push_back((int32_t)j);
      mfirst.push_back((int32_t)nSlots);
      mcount.push_back((int32_t)nseg);
    }
    for (int64_t s = 0; s < nseg; s++) {
      col.push_back((int32_t)j);
      beg.push_back(b + s * SEG);
      len.push_back((int32_t)std::min<int64_t>(SEG, e - (b + s * SEG)));
      slot.push_back(nseg > 1 ? (int32_t)(nSlots + s) : -1);
    }
    if (nseg > 1) nSlots += nseg;
  };
  for (int64_t j = 0; j < d; j++) add_column(j, ptr[(size_t)j], ptr[(size_t)j + 1]);
  for (int a = 0; a < nAug; a++) add_column(d + a, 0, n);   // dummy features: every row, value 1 (dataset.nim:182-189)
  if (nSlots >= (int64_t)1 << 31) return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "too many column segments");
  t->nTasks = (int64_t)col.size();
  t->nMulti = (int64_t)mcol.size();
  t->nSlots = nSlots;
  t->nAug = nAug;
  auto up = [&](auto **dst, const auto &v) -> cudaError_t {
    cudaError_t e = cudaMalloc(dst, std::max<size_t>(v.size(), 1) * sizeof(v[0]));
    if (e == cudaSuccess && !v.empty()) e = cudaMemcpy(*dst, v.data(), v.size() * sizeof(v[0]), cudaMemcpyHostToDevice);
    return e;
  };
  CK(up(&t->taskCol, col));
  CK(up(&t->taskLen, len));
  CK(up(&t->taskSlot, slot));
  CK(up(&t->taskBeg, beg));
  CK(up(&t->multiCol, mcol));
  CK(up(&t->multiFirst, mfirst));
  CK(up(&t->multiCount, mcount));
  guard.t = nullptr;
  *out = t;
  return NIMFM_OK;
}

int nimfm_det_twin_get(nimfm_ctx *ctx, const nimfm_dataset *X, int nAug, nimfm_det_twin **out) {
  if (!X->detTwin || X->detTwin->nAug != nAug) {
    if (X->detTwin) nimfm_det_twin_free(ctx, X->detTwin);
    X->detTwin = nullptr;
    int rc = build_twin(ctx, X, nAug, &X->detTwin);
    if (rc) return rc;
  }
  *out = X->detTwin;
  return NIMFM_OK;
}

// The two passes of the deterministic route over rows [rowBegin, rowBegin + nRows) of X, with the column twin `tw` of
// X (its row ids are X's) and the given targets: the stash forward leaves red4 (loss, sum coef, sum dL^2, -) at
// o.red4, the column kernel and the combine add the gradient into o.gP / o.gw and, when o.gnP is set (AdaGrad, coef =
// dL), its squares into o.gnP / o.gnw.  pl: the stash forward's plan (plan_rows, MODE_STASH); when it is the streaming
// instance the tuned column kernel reads its stash, and every other shape (or NIMFM_ROW_KERNEL=generic, which plans the
// generic stash forward) takes the runtime-k column kernel.  base: the row arguments of X and the model (RowArgs.b may
// point at a refreshed intercept).
int nimfm_fm_det_pass(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_det_twin *tw, const RowPlan &pl, int loss, double thr,
                      int64_t rowBegin, int64_t nRows, double mb, double *yOutDev, const RowArgs &base,
                      const FmDetTargets &o) {
  const bool expl = fm->degree > 2 && fm->nOrders == fm->degree - 1;
  const bool ada = o.gnP != nullptr || o.gnw != nullptr;   // (degree 1 has no P: gnP stays NULL)
  ColKernel ck = nullptr;
  int colKT = fm->k;
  if (fm->nOrders == 0) {   // degree 1: the w-only column pass, one thread per segment
    ck = ada ? fm_cols_linear_kernel<true> : fm_cols_linear_kernel<false>;
    colKT = 1;
  } else if (pl.stream)
    ck = ada ? (fm->degree == 2 ? pick_cols<2, false, true>(fm->k)
                : fm->degree == 3 ? (expl ? pick_cols<3, true, true>(fm->k) : pick_cols<3, false, true>(fm->k)) : nullptr)
             : (fm->degree == 2 ? pick_cols<2, false, false>(fm->k)
                : fm->degree == 3 ? (expl ? pick_cols<3, true, false>(fm->k) : pick_cols<3, false, false>(fm->k)) : nullptr);
  if (!ck) {
    ck = ada ? pick_cols_generic<true>(fm->degree, expl) : pick_cols_generic<false>(fm->degree, expl);
    colKT = lane_group_kt(fm->k);
  }
  if (!ck || !pl.kern)
    return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "no deterministic gradient kernel for degree %d", fm->degree);
  int rc;
  // stash record: coef + (M_o - 1) values per component and order, padded to an even number of doubles
  int vals = 0;
  for (int q = 0; q < fm->nOrders; q++) vals += (fm->degree - q) - 1;
  int stride = 1 + vals * fm->k;
  stride += stride & 1;
  const size_t slotLen = (size_t)(ada ? 2 : 1) * (fm->nOrders * fm->k + 1);
  const size_t need = (size_t)std::max<int64_t>(nRows, 1) * stride + (size_t)tw->nSlots * slotLen + 16;
  if (ctx->stashCap < need) {
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->stash) CK(cudaFree(ctx->stash));
    ctx->stash = nullptr;
    ctx->stashCap = 0;
    if (cudaMalloc(&ctx->stash, need * 8) != cudaSuccess) {
      (void)cudaGetLastError();   // an allocation failure is not sticky: later calls must not see it
      ctx->stash = nullptr;
      return nimfm_fail(ctx, NIMFM_ERR_CUDA,
                        "the deterministic gradient could not allocate its stash: %zu bytes = 8 x (nRows %lld x stride %d "
                        "+ column partial sums); stride = 1 + nComponents x sum_o (degree - o - 1), rounded up to even",
                        need * 8, (long long)nRows, stride);
    }
    ctx->stashCap = need;
  }
  if ((rc = nimfm_ensure_partials(ctx, (size_t)pl.nWarps * 4))) return rc;
  RowArgs a = base;
  a.rowBegin = rowBegin;
  a.nRows = nRows;
  a.rowIdx = nullptr;
  a.yOut = yOutDev;
  a.partials = ctx->partials;
  a.loss = loss;
  a.thr = thr;
  a.mb = mb;
  a.G = pl.G;
  a.CH = pl.CH;
  a.stash = ctx->stash;
  a.stashStride = stride;
  if (o.yhat) a.yOut = o.yhat;
  pl.kern<<<pl.grid, pl.block, pl.smem, ctx->stream>>>(a);
  LAUNCHED(ctx);
  if (o.yhat) {
    const int cgrid = (int)std::max<int64_t>(1, std::min<int64_t>((nRows + 255) / 256, (int64_t)ctx->numSMs * 4));
    if ((rc = nimfm_ensure_partials(ctx, (size_t)cgrid * 4))) return rc;
    dloss_coef_kernel<<<cgrid, 256, 0, ctx->stream>>>(o.yhat, a.y, rowBegin, nRows, loss, thr, mb, ctx->partials);
    LAUNCHED(ctx);
    reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(ctx->partials, cgrid, o.red4, 0);
  } else {
    reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(ctx->partials, pl.nWarps, o.red4, 0);
  }
  LAUNCHED(ctx);
  ColArgs c;
  memset(&c, 0, sizeof(c));
  c.cdata = tw->csc->data;
  c.crow = tw->csc->indices;
  c.taskCol = tw->taskCol;
  c.taskBeg = tw->taskBeg;
  c.taskLen = tw->taskLen;
  c.taskSlot = tw->taskSlot;
  c.nTasks = tw->nTasks;
  c.d = fm->d;
  c.rowBegin = rowBegin;
  c.rowEnd = rowBegin + nRows;
  c.P = fm->P;
  c.stash = ctx->stash;
  c.stashStride = stride;
  c.gP = o.gP;
  c.gw = o.gw;
  c.gnP = o.gnP;
  c.gnw = o.gnw;
  c.partial = ctx->stash + (size_t)std::max<int64_t>(nRows, 1) * stride;
  c.fitLinear = fm->fitLinear;
  c.k = fm->k;
  c.KT = colKT;
  if (tw->nTasks > 0) {
    const int64_t groupsPerBlock = 256 / colKT;
    const int cgrid = (int)std::max<int64_t>(1, std::min<int64_t>((tw->nTasks + groupsPerBlock - 1) / groupsPerBlock,
                                                                  (int64_t)ctx->numSMs * 8));
    ck<<<cgrid, 256, 0, ctx->stream>>>(c);
    LAUNCHED(ctx);
  }
  if (tw->nMulti > 0) {
    const int SB8 = fm->nOrders * fm->k;
    if (ada)
      fm_cols_combine_ada_kernel<<<(unsigned)tw->nMulti, 64, 0, ctx->stream>>>(
          tw->multiCol, tw->multiFirst, tw->multiCount, tw->nMulti, c.partial, SB8, fm->d, c.gP, c.gw, c.gnP, c.gnw,
          fm->fitLinear);
    else
      fm_cols_combine_kernel<<<(unsigned)tw->nMulti, 64, 0, ctx->stream>>>(tw->multiCol, tw->multiFirst, tw->multiCount,
                                                                           tw->nMulti, c.partial, SB8, fm->d, c.gP,
                                                                           c.gw, fm->fitLinear);
    LAUNCHED(ctx);
  }
  CK(cudaGetLastError());
  return NIMFM_OK;
}

// Deterministic predict+grad over rows [rowBegin, rowBegin + nRows) of X into the model's gradient buffers
// (accumulating, like the RED route), with the dataset's column twin.  red4 (loss, sum coef, sum dL^2, -) is left at
// ctx->scalars + 8.
int nimfm_fm_det_loss_grad(nimfm_ctx *ctx, nimfm_fm *fm, const nimfm_dataset *X, const RowPlan &pl, int loss, double thr,
                           int64_t rowBegin, int64_t nRows, double mb, double *yOutDev, const RowArgs &base) {
  if (rowBegin < 0 || rowBegin + nRows > X->n)
    return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "the deterministic gradient needs a contiguous row range without wrap-around");
  int rc;
  nimfm_det_twin *tw = nullptr;
  if ((rc = nimfm_det_twin_get(ctx, X, fm->nAug, &tw))) return rc;
  FmDetTargets o;
  o.gP = fm->grad;
  o.gw = fm->grad + fm->nP();
  o.red4 = ctx->scalars + 8;
  return nimfm_fm_det_pass(ctx, fm, tw, pl, loss, thr, rowBegin, nRows, mb, yOutDev, base, o);
}
