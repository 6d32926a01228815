// ffm_cols.cuh -- FFM predict+grad WITHOUT atomics (included by ffm.cu): forward pair kernel, then a column kernel
// over the CSC twin of the field dataset.
//
// sgd_ffm.nim:23-30 adds, for every pair (u, v) of a row,  dA[f_v][j_u][:] += x_u x_v P[j_v][f_u][:]  (and the
// mirror image).  Read column-wise: the gradient vector of (feature j, field f) is
//     gP[j][f][:] = sum over rows i containing j of  coef_i x_ij  *  sum over the row's nonzeros u of field f,
//                   j_u != j, of  x_iu P[j_u][f_j][:]
// so a block that owns feature j walks j's column entries in ascending row order, thread (f, s) finds the row's
// nonzero of field f through a small position table, gathers ONE k*8-byte vector P[j_u][f_j][:] per (entry,
// field) -- the same bytes the forward pass gathers -- accumulates in a register and finishes with one plain store
// per gradient element (long columns: fixed 512-entry segments, partial sums added in segment order).  Against the
// RED route (ffm_pairs.cuh, 11 856 lane-REDs per 39-field row, each a read-modify-write of a cold line in DRAM)
// this trades 95 KB/row of REDs for a second 95 KB/row of gathers, and every sum has one order: deterministic.
// Needs what the pair route's AdaGrad mode needs -- no row with two nonzeros of one field (checked once per dataset
// on the device) -- and a contiguous row range.  Two column kernels: the tuned ffm_cols_grad_kernel<KT, E> (k in
// {4, 8, 16}, nFields <= 64, rows of at most 64 nonzeros, d * nFields < 2^31) and ffm_cols_grad_generic_kernel<KT, E>
// (every k and nFields, rows of any length, 64-bit offsets), which give the same bits where both run.
#pragma once

struct FfmColArgs {
  const double *cdata;       // CSC twin
  const int32_t *crow;
  const int32_t *taskCol, *taskLen, *taskSlot;
  const int64_t *taskBeg;
  int64_t nTasks;
  const double *data;        // the CSR itself
  const int32_t *indices, *fields;
  const int64_t *indptr;
  const double *coef;        // [rowEnd - rowBegin] coef_i = dloss_i / mb (written by dloss_coef_kernel)
  int64_t rowBegin, rowEnd;
  int nFields, CH;
  int64_t d;
  const double *PT;          // the parameters in FIELD-major layout PT[f][j][s] (see ffm_field_major_kernel)
  double *gP, *gw, *partial;
  int fitLinear;
  int k;                     // ffm_cols_grad_generic_kernel only: nComponents (fills the struct's tail padding)
  double *gnP, *gnw;         // AdaGrad forms: where the squared gradients go (g_norm or its delta block)
};

static __device__ __forceinline__ int64_t lower_bound_row_i32(const int32_t *rows, int64_t lo, int64_t hi, int64_t r) {
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((int64_t)rows[mid] < r) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// columns cut into several segments: their partial sums are added in segment order (one block per column)
static __global__ void ffm_cols_combine_kernel(const int32_t *multiCol, const int32_t *multiFirst, const int32_t *multiCount,
                                               int64_t nMulti, const double *partial, int SB8, double *gP, double *gw,
                                               int fitLinear) {
  const int64_t c = blockIdx.x;
  if (c >= nMulti) return;
  const int64_t j = multiCol[c];
  for (int e = threadIdx.x; e <= SB8; e += blockDim.x) {
    double s = 0.0;
    const double *ps = partial + (size_t)multiFirst[c] * (SB8 + 1) + e;
    for (int q = 0; q < multiCount[c]; ++q) s += ps[(size_t)q * (SB8 + 1)];
    if (e < SB8) gP[j * SB8 + e] += s;
    else if (fitLinear) gw[j] += s;
  }
}

// the AdaGrad form: a slot holds the sums, then the sums of squares, [SB8 | w | SB8 | w]; the second half goes to gnP / gnw
static __global__ void ffm_cols_combine_ada_kernel(const int32_t *multiCol, const int32_t *multiFirst, const int32_t *multiCount,
                                                   int64_t nMulti, const double *partial, int SB8, double *gP, double *gw,
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
    else if (fitLinear) dW[j] += s;
  }
}

// P[j][f][s] (the row kernels' layout: one feature's fields contiguous) -> PT[f][j][s].  The column kernel gathers,
// for a column of field f_j, the vectors P[j_u][f_j][:] of the partner features: in PT they all lie in ONE slab of
// d*k doubles (64 MB for C5) that stays in L2 while the columns of that field are processed, where the row layout
// scatters them over all of P (2.5 GB) -- 64-byte random DRAM accesses, measured at 21 % of the DRAM peak.
static __global__ void ffm_field_major_kernel(const double *P, double *PT, int64_t d, int nF, int k) {
  const int64_t total = d * nF * k;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(e % k);
    const int64_t t = e / k;
    const int64_t j = t % d;
    const int f = (int)(t / d);
    PT[e] = P[(j * nF + f) * k + s];
  }
}

// bytes of shared scratch one warp needs for E entries in flight (must match WarpScratch below)
static inline size_t ffm_cols_warp_smem(int E) {
  const size_t b = (size_t)E * 64 * 8 + (size_t)E * 64 * 4 + (size_t)E * 64 + (size_t)E * 4;
  return (b + 15) & ~(size_t)15;
}

// ONE WARP PER COLUMN SEGMENT, lane <-> field (two passes for nFields > 32), every lane owns the whole k-vector of
// its field in registers.  Per batch of E column entries: lanes < E fetch the entries' row / row pointer / coef*x;
// each entry's row is read with coalesced loads (lane <-> position) into the warp's shared scratch together with
// the inverse table field -> position; then lane f gathers P[j_u][f_j][0..k) for all E entries -- E*k/2 16-byte
// loads in flight per lane -- and accumulates.  No block-wide barrier anywhere: warps run independent segments.
// (The first form -- a block per segment, thread <-> (field, component), three __syncthreads per batch -- ran the
// C5 shape at 21 M rows/s against 60 M for the forward kernel gathering the same bytes: barrier- and latency-bound.)
// ADA (AdaGrad, adagrad.nim:113-124): every product g = sc * v is rounded on its own and g * g is summed into gnP, and
// cx * cx into gnw.  With one nonzero per field, g is the sample's whole gradient element, so its square is the
// reference's.
template <int KT, int E, bool ADA = false>
__global__ void __launch_bounds__(256) ffm_cols_grad_kernel(const FfmColArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int MAXZ = 64;
  struct WarpScratch {
    double x[E][MAXZ];
    int32_t jb[E][MAXZ];
    signed char inv[E][MAXZ];   // field -> position in the row, -1: the row has no nonzero of that field
    int fj[E];
  };
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  WarpScratch &ws = reinterpret_cast<WarpScratch *>(smem_raw)[wib];
  const int nF = a.nFields;
  const int SB8 = nF * KT;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
  const int64_t nWarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t t = warp; t < a.nTasks; t += nWarps) {
    const int64_t j = a.taskCol[t];
    const int32_t jb = (int32_t)(j * nF);
    int64_t eb = a.taskBeg[t], ee = eb + a.taskLen[t];
    if ((int64_t)a.crow[eb] < a.rowBegin) eb = lower_bound_row_i32(a.crow, eb, ee, a.rowBegin);
    if (eb < ee && (int64_t)a.crow[ee - 1] >= a.rowEnd) ee = lower_bound_row_i32(a.crow, eb, ee, a.rowEnd);
    double acc0[KT], acc1[KT], accW = 0.0, accN0[KT], accN1[KT], accWN = 0.0;
#pragma unroll
    for (int c = 0; c < KT; ++c) acc0[c] = acc1[c] = accN0[c] = accN1[c] = 0.0;
    for (int64_t e0 = eb; e0 < ee; e0 += E) {
      const int nb = (int)(ee - e0 < E ? ee - e0 : E);
      int64_t rbL = 0;
      int zL = 0;
      double cxL = 0.0;
      if (lane < nb) {
        const int64_t e = e0 + lane, row = a.crow[e];
        rbL = a.indptr[row];
        zL = (int)(a.indptr[row + 1] - rbL);
        cxL = a.coef[row - a.rowBegin] * a.cdata[e];
      }
      __syncwarp();   // the previous batch's readers are done with the scratch
#pragma unroll
      for (int i = 0; i < E; ++i) {
        ws.inv[i][lane] = -1;
        ws.inv[i][lane + 32] = -1;
      }
      __syncwarp();
      double cx[E];
#pragma unroll
      for (int i = 0; i < E; ++i) {
        const int64_t rb = __shfl_sync(0xffffffffu, rbL, i);
        const int z = __shfl_sync(0xffffffffu, zL, i);
        cx[i] = __shfl_sync(0xffffffffu, cxL, i);
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int u = lane + 32 * half;
          if (i < nb && u < z) {
            const int32_t idx = a.indices[rb + u];
            const int fld = a.fields[rb + u];
            ws.x[i][u] = a.data[rb + u];
            ws.jb[i][u] = idx;
            ws.inv[i][fld] = (signed char)u;
            if (idx == (int32_t)j) ws.fj[i] = fld;
          }
        }
      }
      __syncwarp();
#pragma unroll
      for (int pass = 0; pass < 2; ++pass) {
        const int f = lane + 32 * pass;
        if (pass == 1 && nF <= 32) break;
        double v[E][KT], sc[E];
#pragma unroll
        for (int i = 0; i < E; ++i) {
          sc[i] = 0.0;
#pragma unroll
          for (int c = 0; c < KT; ++c) v[i][c] = 0.0;
          if (i < nb && f < nF) {
            const int u = ws.inv[i][f];
            if (u >= 0 && ws.jb[i][u] != (int32_t)j) {   // the reference pairs distinct features only
              const double2 *src = reinterpret_cast<const double2 *>(a.PT + ((int64_t)ws.fj[i] * a.d + ws.jb[i][u]) * KT);   // P[j_u][f_j][:]
#pragma unroll
              for (int c = 0; c < KT / 2; ++c) {
                const double2 q = __ldg(src + c);
                v[i][2 * c] = q.x;
                v[i][2 * c + 1] = q.y;
              }
              sc[i] = cx[i] * ws.x[i][u];
            }
          }
        }
#pragma unroll
        for (int i = 0; i < E; ++i)   // entries in ascending row order
#pragma unroll
          for (int c = 0; c < KT; ++c) {
            if (ADA) {
              const double g = __dmul_rn(sc[i], v[i][c]);
              if (pass == 0) {
                acc0[c] += g;
                accN0[c] += __dmul_rn(g, g);
              } else {
                acc1[c] += g;
                accN1[c] += __dmul_rn(g, g);
              }
            } else {
              if (pass == 0) acc0[c] += sc[i] * v[i][c];
              else acc1[c] += sc[i] * v[i][c];
            }
          }
      }
      if (lane == 0)
#pragma unroll
        for (int i = 0; i < E; ++i)
          if (i < nb) {
            accW += cx[i];
            if (ADA) accWN += __dmul_rn(cx[i], cx[i]);
          }
    }
    const int slot = a.taskSlot[t];
    double *dst = slot < 0 ? a.gP + (int64_t)jb * KT : a.partial + (size_t)slot * (ADA ? 2 : 1) * (SB8 + 1);
    double *dstN = ADA ? (slot < 0 ? a.gnP + (int64_t)jb * KT : dst + SB8 + 1) : nullptr;
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int f = lane + 32 * pass;
      if (f < nF) {
#pragma unroll
        for (int c = 0; c < KT; ++c) {
          const double val = pass == 0 ? acc0[c] : acc1[c];
          if (slot < 0) dst[f * KT + c] += val;
          else dst[f * KT + c] = val;
          if (ADA) {
            const double valN = pass == 0 ? accN0[c] : accN1[c];
            if (slot < 0) dstN[f * KT + c] += valN;
            else dstN[f * KT + c] = valN;
          }
        }
      }
    }
    if (lane == 0) {
      if (slot < 0) {
        if (a.fitLinear) {
          a.gw[j] += accW;
          if (ADA) a.gnw[j] += accWN;
        }
      } else {
        dst[SB8] = accW;
        if (ADA) dstN[SB8] = accWN;
      }
    }
  }
}

// ffm_cols_grad_kernel with k and nFields at run time.  A task is (column segment, block of 32 fields, component
// chunk of KT); one warp runs one task, lane <-> field fb*32 + lane, KT accumulators per lane.  Per batch of E entries
// the warp reads each entry's row with coalesced loads (lane <-> position, steps of 32), takes the row's own field f_j
// from the position whose feature is j (the lowest such position), and files the positions whose field lies in the
// block as (x, j_u) in a table of 32 field slots: E x 32 x 12 B of shared memory per warp, whatever nFields, k or the
// row length.  The row is read once per (field block, chunk) where the tuned kernel reads it once.  Partner vectors
// come from PT[f_j][j_u][s0 .. s0+KT): 16-byte loads when k is even, scalar loads when it is odd; components past k
// are masked, never read.  Per entry the arithmetic is the tuned kernel's (cx = coef*x_j, sc = cx*x_u, acc += sc*v)
// in the same ascending row order, so where both run they produce the same bits.  ADA: as in ffm_cols_grad_kernel.
template <int KT, int E, bool ADA = false>
__global__ void __launch_bounds__(128) ffm_cols_grad_generic_kernel(const FfmColArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  struct WarpScratch {
    double x[E][32];
    int32_t ju[E][32];   // the feature of the row's nonzero of field fb*32 + slot, -1: none
  };
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  WarpScratch &ws = reinterpret_cast<WarpScratch *>(smem_raw)[wib];
  const int nF = a.nFields, k = a.k;
  const int64_t SB8 = (int64_t)nF * k;
  const int NC = (k + KT - 1) / KT;
  const int64_t per = (int64_t)((nF + 31) >> 5) * NC;
  const int64_t nAll = a.nTasks * per;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + wib;
  const int64_t nWarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t q = warp; q < nAll; q += nWarps) {
    const int64_t t = q / per;
    const int rem = (int)(q - t * per);
    const int fb = rem / NC, s0 = (rem - fb * NC) * KT;
    const int f = fb * 32 + lane;
    const int64_t j = a.taskCol[t];
    int64_t eb = a.taskBeg[t], ee = eb + a.taskLen[t];
    if ((int64_t)a.crow[eb] < a.rowBegin) eb = lower_bound_row_i32(a.crow, eb, ee, a.rowBegin);
    if (eb < ee && (int64_t)a.crow[ee - 1] >= a.rowEnd) ee = lower_bound_row_i32(a.crow, eb, ee, a.rowEnd);
    double acc[KT], accW = 0.0, accN[KT], accWN = 0.0;
#pragma unroll
    for (int c = 0; c < KT; ++c) acc[c] = accN[c] = 0.0;
    for (int64_t e0 = eb; e0 < ee; e0 += E) {
      const int nb = (int)(ee - e0 < E ? ee - e0 : E);
      int64_t rbL = 0;
      int zL = 0;
      double cxL = 0.0;
      if (lane < nb) {
        const int64_t e = e0 + lane, row = a.crow[e];
        rbL = a.indptr[row];
        zL = (int)(a.indptr[row + 1] - rbL);
        cxL = a.coef[row - a.rowBegin] * a.cdata[e];
      }
      __syncwarp();   // the previous batch's readers are done with the scratch
#pragma unroll
      for (int i = 0; i < E; ++i) ws.ju[i][lane] = -1;
      __syncwarp();
      double cx[E];
      int fj[E];
#pragma unroll
      for (int i = 0; i < E; ++i) {
        const int64_t rb = __shfl_sync(0xffffffffu, rbL, i);
        const int z = __shfl_sync(0xffffffffu, zL, i);
        cx[i] = __shfl_sync(0xffffffffu, cxL, i);
        fj[i] = -1;
        for (int u0 = 0; u0 < z; u0 += 32) {   // z is 0 past nb
          const int u = u0 + lane;
          int32_t idx = -1;
          int fld = 0;
          if (u < z) {
            idx = a.indices[rb + u];
            fld = a.fields[rb + u];
            const unsigned slot = (unsigned)(fld - fb * 32);
            if (slot < 32u) {
              ws.x[i][slot] = a.data[rb + u];
              ws.ju[i][slot] = idx;
            }
          }
          const unsigned hit = __ballot_sync(0xffffffffu, idx == (int32_t)j);
          if (hit && fj[i] < 0) fj[i] = __shfl_sync(0xffffffffu, fld, __ffs(hit) - 1);
        }
      }
      __syncwarp();
      double v[E][KT], sc[E];
#pragma unroll
      for (int i = 0; i < E; ++i) {
        sc[i] = 0.0;
#pragma unroll
        for (int c = 0; c < KT; ++c) v[i][c] = 0.0;
        if (i < nb && f < nF && fj[i] >= 0) {
          const int32_t ju = ws.ju[i][lane];
          if (ju >= 0 && ju != (int32_t)j) {   // the reference pairs distinct features only
            const double *src = a.PT + ((int64_t)fj[i] * a.d + ju) * k + s0;   // P[j_u][f_j][s0 ..]
            if ((k & 1) == 0) {   // s0 and k even: 16-byte aligned pairs, both inside k or both past it
#pragma unroll
              for (int c = 0; c < KT / 2; ++c)
                if (s0 + 2 * c < k) {
                  const double2 p = __ldg(reinterpret_cast<const double2 *>(src) + c);
                  v[i][2 * c] = p.x;
                  v[i][2 * c + 1] = p.y;
                }
            } else {
#pragma unroll
              for (int c = 0; c < KT; ++c)
                if (s0 + c < k) v[i][c] = __ldg(src + c);
            }
            sc[i] = cx[i] * ws.x[i][lane];
          }
        }
      }
#pragma unroll
      for (int i = 0; i < E; ++i)   // entries in ascending row order
#pragma unroll
        for (int c = 0; c < KT; ++c) {
          if (ADA) {
            const double g = __dmul_rn(sc[i], v[i][c]);
            acc[c] += g;
            accN[c] += __dmul_rn(g, g);
          } else {
            acc[c] += sc[i] * v[i][c];
          }
        }
      if (lane == 0)
#pragma unroll
        for (int i = 0; i < E; ++i)
          if (i < nb) {
            accW += cx[i];
            if (ADA) accWN += __dmul_rn(cx[i], cx[i]);
          }
    }
    const int slot = a.taskSlot[t];
    double *dst = slot < 0 ? a.gP + j * SB8 : a.partial + (size_t)slot * (ADA ? 2 : 1) * (SB8 + 1);
    double *dstN = ADA ? (slot < 0 ? a.gnP + j * SB8 : dst + SB8 + 1) : nullptr;
    if (f < nF) {
#pragma unroll
      for (int c = 0; c < KT; ++c) {
        if (s0 + c >= k) break;
        if (slot < 0) dst[(int64_t)f * k + s0 + c] += acc[c];
        else dst[(int64_t)f * k + s0 + c] = acc[c];
        if (ADA) {
          if (slot < 0) dstN[(int64_t)f * k + s0 + c] += accN[c];
          else dstN[(int64_t)f * k + s0 + c] = accN[c];
        }
      }
    }
    if (lane == 0 && fb == 0 && s0 == 0) {   // one task per segment owns the linear term
      if (slot < 0) {
        if (a.fitLinear) {
          a.gw[j] += accW;
          if (ADA) a.gnw[j] += accWN;
        }
      } else {
        dst[SB8] = accW;
        if (ADA) dstN[SB8] = accWN;
      }
    }
  }
}

// the component chunk of ffm_cols_grad_generic_kernel: lanes map to fields, so there are no idle lanes to weigh; the
// narrowest width that holds k in one chunk wastes the fewest accumulator registers, and k > 32 takes chunks of 32
// (the widest instance that does not spill)
static inline int ffm_cols_generic_kt(int k) { return k <= 4 ? 4 : k <= 8 ? 8 : k <= 16 ? 16 : 32; }

// bytes of shared scratch one warp of ffm_cols_grad_generic_kernel<KT, E> needs (must match its WarpScratch)
static inline size_t ffm_cols_generic_warp_smem(int E) { return (size_t)E * 32 * (8 + 4); }
