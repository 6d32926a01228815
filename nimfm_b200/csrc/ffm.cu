// ffm.cu -- FieldAwareFactorizationMachine on the device (SURVEY K10, K11, a14, a15):
// decisionFunction (model/field_aware_factorization_machine.nim:52-76), predict+grad
// (optimizer/sgd_ffm.nim:11-30) and minibatch AdaGrad (optimizer/adagrad_ffm.nim:11-66 over
// adagrad.nim:87-134 with "order" == field).
//
// Device layout P[j][f][s]: the nFields*k doubles one feature owns are contiguous (2496 B for
// 39 fields x rank 8), versus the reference's P[f][j][s] where they are nFeatures*k*8 bytes apart.
//
// Kernel: ONE THREAD BLOCK PER ROW.  The block stages the row's z feature slices W[u][f][s]
// (z * nFields * k doubles, 97 KB for the C5 shape) in shared memory with cp.async, buckets the
// row's nonzeros by field, and evaluates for every entry (u, f, s)
//     dA[u][f][s] = x_u * sum_{v in bucket f, v != u} x_v * W[v][f_u][s]          (sgd_ffm.nim:23-30)
// from shared memory.  The pair sum of the forward pass is 1/2 sum_{u,f,s} W[u][f][s]*dA[u][f][s]
// (every unordered pair {u,v}, j_u != j_v, is counted once from each side), so forward and
// backward are two sweeps of the same loop; the backward sweep emits coef*dA with FP64 RED atomics
// (entries whose field bucket is empty have dA == 0 and are skipped).
#include <math.h>

#include <algorithm>

#include "dense_kernels.cuh"

enum { FFM_PREDICT = 0, FFM_GRAD = 1, FFM_ADAGRAD = 2 };

#define FFM_THREADS 256

struct FfmArgs {
  const double *data;
  const int32_t *indices, *fields;
  const int64_t *indptr;
  const double *y;
  int64_t n, rowBegin, nRows;
  const int32_t *rowIdx;
  int k, nFields;
  int64_t d;
  const double *P, *w, *b;
  int fitLinear, fitIntercept;
  double *yOut, *gP, *gw, *partials;   // partials: [gridDim][4] loss, sum coef | sum dL, sum dL^2, viol
  int loss;
  double thr, mb;
  const double *gsP, *gnP, *gsw, *gnw, *adaScal;
  double *dGnP, *dGnw, *touched;
  double eta0, tIt, alpha0, alpha, beta;
  int first;
  int CH;   // staging capacity in nonzeros (>= longest row)
  unsigned char *unitScratch;   // ffm_units_kernel: per-block records of rows past FFM_UNITS_SMEM_CAP (nimfm_ffm)
};

struct __align__(16) FfmMeta {
  double x;
  int32_t j;
  int32_t f;
};

#include "ffm_pairs.cuh"
#include "ffm_cols.cuh"
#include "ffm_units.cuh"

static size_t ffm_smem_bytes(int CH, int SB8, int nFields) {
  size_t b = (((size_t)CH * SB8 * 8 + 15) & ~(size_t)15) + (size_t)CH * sizeof(FfmMeta) + (size_t)CH * 4 +
             (size_t)(nFields + 1) * 4 * 2;
  return (b + 15) & ~(size_t)15;
}

template <int MODE>
__global__ void __launch_bounds__(FFM_THREADS, 1) ffm_rows_kernel(const FfmArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double red[FFM_THREADS / 32];
  __shared__ double shv[2];
  const int k = a.k, nF = a.nFields, SB8 = nF * k, CH = a.CH;
  double *sW = reinterpret_cast<double *>(smem_raw);
  FfmMeta *sMeta = reinterpret_cast<FfmMeta *>(smem_raw + ((((size_t)CH * SB8 * 8) + 15) & ~(size_t)15));
  int *sOrd = reinterpret_cast<int *>(sMeta + CH);
  int *sStart = sOrd + CH;          // [nF + 1]
  int *sCursor = sStart + nF + 1;   // [nF + 1]
  const int tid = threadIdx.x, nth = blockDim.x;
  double accLoss = 0.0, accB1 = 0.0, accB2 = 0.0, accViol = 0.0;
  double bias = a.b[0];
  if (MODE == FFM_ADAGRAD) {
    if (!a.first && a.fitIntercept) {
      const double den = sqrt(a.adaScal[1]) + a.eta0 * a.tIt * a.alpha0;
      bias = -a.eta0 * a.adaScal[0] / den;
    }
  }

  for (int64_t q = blockIdx.x; q < a.nRows; q += gridDim.x) {
    const int64_t r = a.rowIdx ? (int64_t)a.rowIdx[q] : (a.rowBegin + q) % a.n;
    const int64_t rb = a.indptr[r];
    const int z = (int)(a.indptr[r + 1] - rb);
    __syncthreads();
    // ---- metadata, linear term, field buckets
    for (int f = tid; f <= nF; f += nth) sStart[f] = 0;
    __syncthreads();
    double lin = 0.0;
    for (int u = tid; u < z; u += nth) {
      FfmMeta m;
      m.j = a.indices[rb + u];
      m.f = a.fields[rb + u];
      m.x = a.data[rb + u];
      sMeta[u] = m;
      atomicAdd(&sStart[m.f + 1], 1);
      lin += a.w[m.j] * m.x;
    }
    __syncthreads();
    if (tid == 0) {
      for (int f = 0; f < nF; f++) sStart[f + 1] += sStart[f];
      for (int f = 0; f <= nF; f++) sCursor[f] = sStart[f];
      // stable by position: serial fill keeps the order deterministic (rows are short)
      for (int u = 0; u < z; u++) sOrd[sCursor[sMeta[u].f]++] = u;
    }
    // ---- stage W = the row's feature slices (AdaGrad: P was refreshed by adagrad_refresh_kernel)
    {
      if ((SB8 & 1) == 0) {
        const int units = SB8 >> 1, total = z * units;
        for (int v = tid; v < total; v += nth) {
          const int qq = v / units, off = (v - qq * units) << 1;
          cp_async16(sW + (size_t)qq * SB8 + off, a.P + (int64_t)sMeta[qq].j * SB8 + off);
        }
      } else {
        const int total = z * SB8;
        for (int v = tid; v < total; v += nth) {
          const int qq = v / SB8, off = v - qq * SB8;
          cp_async8(sW + (size_t)qq * SB8 + off, a.P + (int64_t)sMeta[qq].j * SB8 + off);
        }
      }
      cp_async_wait_all();
    }
    __syncthreads();

    // ---- sweep 1: forward
    double part = 0.0;
    for (int e = tid; e < z * SB8; e += nth) {
      const int u = e / SB8, fs = e - u * SB8;
      const int f = fs / k, s = fs - f * k;
      const int b0 = sStart[f], b1 = sStart[f + 1];
      if (b0 == b1) continue;
      const FfmMeta mu = sMeta[u];
      double acc = 0.0;
      for (int t = b0; t < b1; ++t) {
        const int v = sOrd[t];
        if (v != u) acc += sMeta[v].x * sW[(size_t)v * SB8 + mu.f * k + s];
      }
      part += sW[e] * (mu.x * acc);
    }
    double tot = block_sum(lin + 0.5 * part, red);
    if (tid == 0) {
      const double yhat = bias + tot;
      if (a.yOut) a.yOut[q] = yhat;
      double dL = 0.0;
      if (MODE != FFM_PREDICT) {
        const double yi = a.y[r];
        dL = dev_dloss(a.loss, a.thr, yi, yhat);
        accLoss += dev_loss(a.loss, a.thr, yi, yhat);
        const double coef = MODE == FFM_GRAD ? dL / a.mb : dL;
        accB1 += coef;
        accB2 += dL * dL;
        shv[0] = coef;
      }
    }
    if (MODE == FFM_PREDICT) continue;
    __syncthreads();
    const double coef = shv[0];

    // ---- sweep 2: gradient scatter
    for (int e = tid; e < z * SB8; e += nth) {
      const int u = e / SB8, fs = e - u * SB8;
      const int f = fs / k, s = fs - f * k;
      const int b0 = sStart[f], b1 = sStart[f + 1];
      if (b0 == b1) continue;
      const FfmMeta mu = sMeta[u];
      double acc = 0.0;
      for (int t = b0; t < b1; ++t) {
        const int v = sOrd[t];
        if (v != u) acc += sMeta[v].x * sW[(size_t)v * SB8 + mu.f * k + s];
      }
      const double gr = coef * (mu.x * acc);
      if (gr != 0.0) {
        const int64_t ge = (int64_t)mu.j * SB8 + fs;
        atomicAdd(a.gP + ge, gr);
        if (MODE == FFM_ADAGRAD) atomicAdd(a.dGnP + ge, gr * gr);
      }
    }
    for (int u = tid; u < z; u += nth) {
      const FfmMeta m = sMeta[u];
      if (a.fitLinear) {
        const double gx = coef * m.x;
        atomicAdd(a.gw + m.j, gx);
        if (MODE == FFM_ADAGRAD) atomicAdd(a.dGnw + m.j, gx * gx);
      }
    }
  }

  if (MODE != FFM_PREDICT) {
    __syncthreads();
    accViol = block_sum(accViol, red);
    __syncthreads();
    if (tid == 0) {
      a.partials[blockIdx.x * 4 + 0] = accLoss;
      a.partials[blockIdx.x * 4 + 1] = accB1;
      a.partials[blockIdx.x * 4 + 2] = accB2;
      a.partials[blockIdx.x * 4 + 3] = accViol;
    }
  }
}

// ------------------------------------------------------------------ layout: reference P[f][j][s] <-> device P[j][f][s]
static __global__ void ffm_permute_kernel(const double *R, double *D, int64_t nF, int64_t d, int k, int toDev) {
  const int64_t total = nF * d * k;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int s = (int)(e % k);
    const int64_t t = e / k;
    const int64_t f = t % nF, j = t / nF;            // e indexes the device layout
    const int64_t re = (f * d + j) * k + s;
    if (toDev) D[e] = R[re];
    else const_cast<double *>(R)[re] = D[e];
  }
}

typedef void (*FfmKernel)(const FfmArgs);

struct FfmPlan {
  int CH, grid;
  size_t smem;
  FfmKernel kern = nullptr;
  int block = FFM_THREADS;
  int64_t partialRows = 0;   // rows of the [.][4] partials block the kernel writes
};

// pair-streaming kernel when k is 4/8/16/32, else nullptr
template <int KT>
static FfmKernel ffm_pairs_mode(int mode) {
  return mode == FFM_PREDICT ? ffm_pairs_kernel<FFM_PAIRS_PREDICT, KT, FfmArgs>
         : mode == FFM_GRAD  ? ffm_pairs_kernel<FFM_PAIRS_GRAD, KT, FfmArgs>
                             : ffm_pairs_kernel<FFM_PAIRS_ADAGRAD, KT, FfmArgs>;
}
static FfmKernel ffm_pairs_pick(int k, int mode) {
  switch (k) {
    case 4: return ffm_pairs_mode<4>(mode);
    case 8: return ffm_pairs_mode<8>(mode);
    case 16: return ffm_pairs_mode<16>(mode);
    case 32: return ffm_pairs_mode<32>(mode);
    default: return nullptr;
  }
}

template <int KT>
static FfmKernel ffm_pairs_block_mode(int mode) {
  return mode == FFM_PREDICT ? ffm_pairs_block_kernel<FFM_PAIRS_PREDICT, KT, FfmArgs>
         : mode == FFM_GRAD  ? ffm_pairs_block_kernel<FFM_PAIRS_GRAD, KT, FfmArgs>
                             : ffm_pairs_block_kernel<FFM_PAIRS_ADAGRAD, KT, FfmArgs>;
}
static FfmKernel ffm_pairs_block_pick(int k, int mode) {
  switch (k) {
    case 4: return ffm_pairs_block_mode<4>(mode);
    case 8: return ffm_pairs_block_mode<8>(mode);
    case 16: return ffm_pairs_block_mode<16>(mode);
    case 32: return ffm_pairs_block_mode<32>(mode);
    default: return nullptr;
  }
}

template <int KT>
static FfmKernel ffm_pairs_bulk_mode(int mode) {
  return mode == FFM_GRAD      ? ffm_pairs_block_kernel<FFM_PAIRS_GRAD, KT, FfmArgs, true>
         : mode == FFM_ADAGRAD ? ffm_pairs_block_kernel<FFM_PAIRS_ADAGRAD, KT, FfmArgs, true>
                               : nullptr;
}
static FfmKernel ffm_pairs_bulk_pick(int k, int mode) {
  switch (k) {
    case 4: return ffm_pairs_bulk_mode<4>(mode);
    case 8: return ffm_pairs_bulk_mode<8>(mode);
    case 16: return ffm_pairs_bulk_mode<16>(mode);
    case 32: return ffm_pairs_bulk_mode<32>(mode);
    default: return nullptr;
  }
}

// does any row hold two nonzeros of one field?  (computed once per dataset, on the device)
static int ffm_has_field_dups(nimfm_ctx *ctx, const nimfm_dataset *X, bool *dups) {
  if (X->fieldDup < 0) {
    int *flag = nullptr;
    CK(cudaMalloc(&flag, sizeof(int)));
    CK(cudaMemsetAsync(flag, 0, sizeof(int), ctx->stream));
    if (X->n > 0) {
      const int grid = (int)std::min<int64_t>((X->n * 32 + 255) / 256, (int64_t)ctx->numSMs * 16);
      ffm_field_dup_kernel<<<grid < 1 ? 1 : grid, 256, 0, ctx->stream>>>(X->fields, X->indptr, X->n, flag);
      LAUNCHED(ctx);
    }
    int h = 0;
    CK(cudaMemcpyAsync(&h, flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaFree(flag));
    X->fieldDup = h ? 1 : 0;
  }
  *dups = X->fieldDup == 1;
  return NIMFM_OK;
}

static int ffm_plan(nimfm_ctx *ctx, const nimfm_ffm *m, const nimfm_dataset *X, int64_t nRows, FfmKernel kern,
                    FfmPlan *pl, bool *declined);

template <int KT>
static FfmKernel ffm_units_mode(int mode) {
  return mode == FFM_PREDICT ? ffm_units_kernel<FFM_PREDICT, KT>
         : mode == FFM_GRAD  ? ffm_units_kernel<FFM_GRAD, KT>
                             : ffm_units_kernel<FFM_ADAGRAD, KT>;
}
static FfmKernel ffm_units_pick(int k, int mode) {
  switch (lane_group_kt(k)) {
    case 4: return ffm_units_mode<4>(mode);
    case 8: return ffm_units_mode<8>(mode);
    case 16: return ffm_units_mode<16>(mode);
    default: return ffm_units_mode<32>(mode);
  }
}

// global scratch of the unit kernel's long rows (ffm_units_row_bytes(longest row) per block) is held to this many
// bytes by shrinking the grid
#define FFM_UNITS_SCRATCH_MAX ((size_t)256 << 20)

// the (nonzero, field) kernel (ffm_units.cuh): any k, any row length
static int ffm_plan_units(nimfm_ctx *ctx, const nimfm_ffm *m, const nimfm_dataset *X, int64_t nRows, int mode,
                          FfmPlan *pl) {
  const int CH = (int)std::max<int64_t>(X->maxSegNnz, 1);
  FfmKernel kern = ffm_units_pick(m->k, mode);
  const size_t smem = ffm_units_row_bytes(std::min(CH, FFM_UNITS_SMEM_CAP));
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, FFM_UNITS_THREADS, smem));
  if (occ < 1) return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "FFM unit kernel does not fit on an SM");
  int64_t grid = std::min<int64_t>(nRows, (int64_t)occ * ctx->numSMs);
  if (grid < 1) grid = 1;
  if (CH > FFM_UNITS_SMEM_CAP) {
    const size_t rowBytes = ffm_units_row_bytes(CH);
    grid = std::max<int64_t>(1, std::min<int64_t>(grid, (int64_t)(FFM_UNITS_SCRATCH_MAX / rowBytes)));
    const size_t need = (size_t)grid * rowBytes;
    if (m->unitScratchBytes < need) {
      CK(cudaStreamSynchronize(ctx->stream));   // an earlier launch may still read the old area
      CK(cudaFree(m->unitScratch));
      m->unitScratch = nullptr;
      m->unitScratchBytes = 0;
      CK(cudaMalloc(&m->unitScratch, need));
      m->unitScratchBytes = need;
    }
  }
  pl->CH = CH;
  pl->grid = (int)grid;
  pl->smem = smem;
  pl->kern = kern;
  pl->block = FFM_UNITS_THREADS;
  pl->partialRows = grid;
  return NIMFM_OK;
}

// Every mode chooses a pair kernel when one exists for k (NIMFM_FFM_KERNEL=block forces the staged
// block-per-row kernel ffm_rows_kernel); FFM_ADAGRAD additionally needs a dataset without repeated
// fields in a row.  The staged kernel takes the rest; where its row does not fit shared memory, the
// (nonzero, field) kernel ffm_units_kernel does (NIMFM_FFM_KERNEL=units forces it for every shape).
static int ffm_plan_mode(nimfm_ctx *ctx, const nimfm_ffm *m, const nimfm_dataset *X, int64_t nRows, int mode,
                         FfmPlan *pl, bool targetsAligned16 = true) {
  const char *env = getenv("NIMFM_FFM_KERNEL");
  const bool forceBlock = env && !strcmp(env, "block");
  if (env && !strcmp(env, "units")) return ffm_plan_units(ctx, m, X, nRows, mode, pl);
  const int CH = (int)std::max<int64_t>(X->maxSegNnz, 1);
  const bool table = CH <= FFM_PAIRS_TABLE_MAXZ;
  // the pair kernel addresses P through 32-bit (j*nFields + f): needs d*nFields < 2^31
  FfmKernel pk = (forceBlock || CH > 1024 || m->d * m->nFields >= (int64_t)2147483647)
                     ? nullptr : ffm_pairs_pick(m->k, mode);
  if (pk && mode == FFM_ADAGRAD) {
    // the pair kernel squares per-pair contributions, which equals the per-sample gradient entry
    // (adagrad.nim:119-124) only when no row has two nonzeros of one field
    bool dups = false;
    int rc = ffm_has_field_dups(ctx, X, &dups);
    if (rc) return rc;
    if (dups) pk = nullptr;
  }
  // Gradient blocks assembled in shared memory and added by TMA bulk reductions (ffm_pairs.cuh); needs a dataset
  // without repeated fields in a row (every segment of a block is written by exactly one partner).  Default for
  // the AdaGrad mode (two reductions per nonzero instead of 2 x 370 warp REDs per row: 13.3 -> 14.8 M samples/s on
  // C5); predict+grad runs at the L2's FP64-add rate either way (22.3 M rows/s RED, 21.2 M bulk) and keeps the
  // REDs.  NIMFM_FFM_BULK=0/1 forces either.
  const char *benv = getenv("NIMFM_FFM_BULK");
  const bool wantBulk = benv ? atoi(benv) == 1 : mode == FFM_ADAGRAD;
  // a bulk reduction wants 16-byte aligned global targets: an even block length and aligned buffer bases
  if (pk && table && mode != FFM_PREDICT && wantBulk && ((m->nFields * m->k) & 1) == 0 &&
      targetsAligned16) {
    bool dups = false;
    int rc = ffm_has_field_dups(ctx, X, &dups);
    if (rc) return rc;
    FfmKernel bk = dups ? nullptr : ffm_pairs_bulk_pick(m->k, mode);
    const int block = 256;
    const size_t smem = ffm_bulk_smem(CH, (int)(m->nFields * m->k), mode == FFM_ADAGRAD ? 2 : 1, block / 32);
    if (bk && smem <= (size_t)ctx->smemOptin) {
      CK(cudaFuncSetAttribute(bk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      int occ = 0;
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bk, block, smem));
      if (occ >= 1) {
        int64_t grid = std::min<int64_t>(nRows, (int64_t)occ * ctx->numSMs);
        if (grid < 1) grid = 1;
        pl->CH = CH;
        pl->grid = (int)grid;
        pl->smem = smem;
        pl->kern = bk;
        pl->block = block;
        pl->partialRows = grid;
        return NIMFM_OK;
      }
    }
  }
  // rows up to FFM_PAIRS_TABLE_MAXZ nonzeros: the block-per-row form of the pair loop (grad 15.1 -> 22.7 M
  // rows/s on C5); longer rows take the warp-per-row form
  if (pk && table) {
    FfmKernel bk = ffm_pairs_block_pick(m->k, mode);
    const int block = 256;
    const size_t smem = ffm_pairs_warp_smem(CH, true);
    CK(cudaFuncSetAttribute(bk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, bk, block, smem));
    if (occ < 1) return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "FFM pair-block kernel does not fit on an SM");
    int64_t grid = std::min<int64_t>(nRows, (int64_t)occ * ctx->numSMs);
    if (grid < 1) grid = 1;
    pl->CH = CH;
    pl->grid = (int)grid;
    pl->smem = smem;
    pl->kern = bk;
    pl->block = block;
    pl->partialRows = grid;
    return NIMFM_OK;
  }
  if (pk) {
    const int block = 256, wpb = block / 32;
    const size_t smem = (size_t)wpb * ffm_pairs_warp_smem(CH, false);
    CK(cudaFuncSetAttribute(pk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pk, block, smem));
    if (occ < 1) return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "FFM pair kernel does not fit on an SM");
    int64_t grid = std::min<int64_t>((nRows + wpb - 1) / wpb, (int64_t)occ * ctx->numSMs);
    if (grid < 1) grid = 1;
    pl->CH = CH;
    pl->grid = (int)grid;
    pl->smem = smem;
    pl->kern = pk;
    pl->block = block;
    pl->partialRows = grid * wpb;
    return NIMFM_OK;
  }
  FfmKernel bk = mode == FFM_PREDICT ? ffm_rows_kernel<FFM_PREDICT>
                 : mode == FFM_GRAD  ? ffm_rows_kernel<FFM_GRAD>
                                     : ffm_rows_kernel<FFM_ADAGRAD>;
  bool declined = false;
  int rc = ffm_plan(ctx, m, X, nRows, bk, pl, forceBlock ? nullptr : &declined);
  if (rc) return rc;
  if (declined) return ffm_plan_units(ctx, m, X, nRows, mode, pl);
  pl->kern = bk;
  pl->block = FFM_THREADS;
  pl->partialRows = pl->grid;
  return NIMFM_OK;
}

// declined != nullptr: a shape the staged kernel cannot run sets *declined instead of failing
static int ffm_plan(nimfm_ctx *ctx, const nimfm_ffm *m, const nimfm_dataset *X, int64_t nRows, FfmKernel kern,
                    FfmPlan *pl, bool *declined) {
  const int SB8 = (int)(m->nFields * m->k);
  const int CH = (int)std::max<int64_t>(X->maxSegNnz, 1);
  const size_t smem = ffm_smem_bytes(CH, SB8, (int)m->nFields);
  if (smem > (size_t)ctx->smemOptin) {
    if (declined) { *declined = true; return NIMFM_OK; }
    return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED,
                      "FFM row of %d nonzeros x %d fields x rank %d needs %zu B of shared memory (> %d)", CH,
                      (int)m->nFields, m->k, smem, ctx->smemOptin);
  }
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, FFM_THREADS, smem));
  if (occ < 1) {
    if (declined) { *declined = true; return NIMFM_OK; }
    return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "FFM kernel does not fit on an SM");
  }
  int64_t grid = std::min<int64_t>(nRows, (int64_t)occ * ctx->numSMs);
  if (grid < 1) grid = 1;
  pl->CH = CH;
  pl->grid = (int)grid;
  pl->smem = smem;
  return NIMFM_OK;
}

static int check_ffm_ds(nimfm_ctx *ctx, const nimfm_ffm *m, const nimfm_dataset *X, bool needY) {
  REQUIRE(m && X, "NULL handle");
  REQUIRE(X->kind == NIMFM_DS_CSR_FIELD, "a CSRFieldDataset is required");
  REQUIRE(X->d == m->d, "Invalid nFeatures.");        // field_aware_factorization_machine.nim:60-61
  REQUIRE(X->nFields == m->nFields, "Invalid nFields.");  // :62-64
  REQUIRE(!needY || X->y != nullptr, "dataset has no targets (nimfm_dataset_set_targets)");
  return NIMFM_OK;
}

static void ffm_fill_args(FfmArgs &a, const nimfm_ffm *m, const nimfm_dataset *X) {
  memset(&a, 0, sizeof(a));
  a.data = X->data; a.indices = X->indices; a.fields = X->fields; a.indptr = X->indptr; a.y = X->y;
  a.n = X->n;
  a.k = m->k; a.nFields = (int)m->nFields; a.d = m->d;
  a.P = m->P; a.w = m->w; a.b = m->b;
  a.fitLinear = m->fitLinear; a.fitIntercept = m->fitIntercept;
  a.mb = 1.0;
  a.unitScratch = m->unitScratch;
}

extern "C" {

int32_t nimfm_ffm_create(nimfm_ctx *ctx, int32_t nComponents, int64_t nFields, int64_t nFeatures,
                         int32_t fitLinear, int32_t fitIntercept, nimfm_ffm **out) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(out != nullptr, "out is NULL");
  REQUIRE(nComponents >= 1, "nComponents < 1.");
  REQUIRE(nFields >= 1 && nFeatures >= 1, "nFields / nFeatures < 1");
  CK(cudaSetDevice(ctx->device));
  nimfm_ffm *m = new nimfm_ffm();
  m->k = nComponents; m->nFields = nFields; m->d = nFeatures;
  m->fitLinear = fitLinear != 0; m->fitIntercept = fitIntercept != 0;
  const int64_t nP = m->nP();
  CK(cudaMalloc(&m->P, (size_t)nP * 8));
  CK(cudaMalloc(&m->w, (size_t)m->d * 8));
  CK(cudaMalloc(&m->b, 8 * 8));
  { int rca = nimfm_comm_alloc(ctx, &m->grad, (size_t)(nP + m->d + 2)); if (rca) { nimfm_ffm_free(ctx, m); return rca; } }
  CK(cudaMemsetAsync(m->P, 0, (size_t)nP * 8, ctx->stream));
  CK(cudaMemsetAsync(m->w, 0, (size_t)m->d * 8, ctx->stream));
  CK(cudaMemsetAsync(m->b, 0, 64, ctx->stream));
  CK(cudaMemsetAsync(m->grad, 0, (size_t)(nP + m->d + 2) * 8, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  *out = m;
  return NIMFM_OK;
}

int32_t nimfm_ffm_free(nimfm_ctx *ctx, nimfm_ffm *m) {
  if (!m) return NIMFM_OK;
  if (ctx) cudaSetDevice(ctx->device);
  nimfm_comm_free(ctx, m->grad);
  nimfm_comm_free(ctx, m->dG);
  nimfm_comm_free(ctx, m->sgdCnt);
  for (double *p : {m->P, m->PT, m->w, m->b, m->gsP, m->gnP, m->gsw, m->gnw, m->adaScal, m->scalingsP,
                    m->scalingsW, m->sgdScal})
    cudaFree(p);
  cudaFree(m->unitScratch);
  delete m;
  return NIMFM_OK;
}

static int ffm_permute(nimfm_ctx *ctx, nimfm_ffm *m, double *host, double *dev, int toDev) {
  const int64_t nP = m->nP();
  double *tmp = nullptr;
  CK(cudaMalloc(&tmp, (size_t)nP * 8));
  if (toDev) { int rcs = nimfm_staged_h2d(ctx, tmp, host, (size_t)nP * 8); if (rcs) { cudaFree(tmp); return rcs; } }
  ffm_permute_kernel<<<ew_grid(ctx, nP), 256, 0, ctx->stream>>>(tmp, dev, m->nFields, m->d, m->k, toDev);
  LAUNCHED(ctx);
  if (!toDev) { int rcs = nimfm_staged_d2h(ctx, host, tmp, (size_t)nP * 8); if (rcs) { cudaFree(tmp); return rcs; } }
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaFree(tmp));
  CK(cudaGetLastError());
  return NIMFM_OK;
}

int32_t nimfm_ffm_set_params(nimfm_ctx *ctx, nimfm_ffm *m, const double *P, const double *w, double intercept) {
  if (!ctx || !m) return NIMFM_ERR_INVALID;
  REQUIRE(P && w, "P / w are NULL");
  CK(cudaSetDevice(ctx->device));
  int rc = ffm_permute(ctx, m, const_cast<double *>(P), m->P, 1);
  if (rc) return rc;
  CK(cudaMemcpy(m->w, w, (size_t)m->d * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(m->b, &intercept, 8, cudaMemcpyHostToDevice));
  return NIMFM_OK;
}

int32_t nimfm_ffm_get_params(nimfm_ctx *ctx, nimfm_ffm *m, double *P, double *w, double *intercept) {
  if (!ctx || !m) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int rc;
  if (P && (rc = ffm_permute(ctx, m, P, m->P, 0))) return rc;
  if (w) CK(cudaMemcpy(w, m->w, (size_t)m->d * 8, cudaMemcpyDeviceToHost));
  if (intercept) CK(cudaMemcpy(intercept, m->b, 8, cudaMemcpyDeviceToHost));
  return NIMFM_OK;
}

int32_t nimfm_ffm_get_grads(nimfm_ctx *ctx, nimfm_ffm *m, double *gP, double *gw, double *gb) {
  if (!ctx || !m) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int rc;
  if (gP && (rc = ffm_permute(ctx, m, gP, m->grad, 0))) return rc;
  if (gw) CK(cudaMemcpy(gw, m->grad + m->nP(), (size_t)m->d * 8, cudaMemcpyDeviceToHost));
  if (gb) CK(cudaMemcpy(gb, m->grad + m->nP() + m->d, 8, cudaMemcpyDeviceToHost));
  return NIMFM_OK;
}

// K10
int32_t nimfm_ffm_decision_function(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, double *out) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int rc = check_ffm_ds(ctx, m, X, false);
  if (rc) return rc;
  REQUIRE(out != nullptr, "out is NULL");
  const int64_t n = X->n;
  if (n == 0) return NIMFM_OK;
  FfmPlan pl;
  if ((rc = ffm_plan_mode(ctx, m, X, n, FFM_PREDICT, &pl))) return rc;
  double *dOut = nullptr;
  CK(cudaMalloc(&dOut, (size_t)n * 8));
  FfmArgs a;
  ffm_fill_args(a, m, X);
  a.nRows = n;
  a.yOut = dOut;
  a.CH = pl.CH;
  pl.kern<<<pl.grid, pl.block, pl.smem, ctx->stream>>>(a);
  LAUNCHED(ctx);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, dOut, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaFree(dOut));
  return NIMFM_OK;
}

// The atomic-free route (ffm_cols.cuh), taken under NIMFM_DETERMINISTIC=1: every contiguous row range of a dataset
// without repeated fields runs, with the tuned column kernel where its shape limits hold and the generic one elsewhere;
// any other request is an error.  NIMFM_FFM_COLS=generic puts the generic kernel in the tuned kernel's place.
// A stated upper bound on the generic column kernel's resident 128-thread blocks per SM, not a tuning choice: it
// equals the register-limited occupancy of the 112 / 126-register instances and lies above that of the 200 /
// 225-register ones (2), so it changes no launch; the tests size their data past three waves of this bound.
#define FFM_COLS_GENERIC_BLOCKS_PER_SM 4
// where the column route's outputs go (ffm_det_pass)
struct FfmDetTargets {
  double *gP, *gw;       // gradient sums (the model's gradient, g_sum or its delta block)
  double *gnP, *gnw;     // AdaGrad: sums of squared gradients; nullptr: plain gradient
  double *red4;          // (loss, sum coef, sum dL^2, -)
  const double *b;       // the intercept the forward pass sees
};

// AdaGrad's generic column-kernel width: ffm_cols_generic_kt, but k > 16 takes chunks of 16 -- the square accumulators
// do not fit beside 32 components per lane without spills (ptxas)
static inline int ffm_cols_ada_kt(int k) { return k <= 4 ? 4 : k <= 8 ? 8 : 16; }

// the two passes of the column route over rows [rowBegin, rowBegin + nRows) of X with X's column twin tw (row ids
// X's): the forward kernel and dloss_coef_kernel, then the tuned column kernel (tunedKernel) or the generic one
static int ffm_det_pass(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, const nimfm_det_twin *tw, int loss,
                        double thr, int64_t rowBegin, int64_t nRows, double mb, bool tunedKernel,
                        const FfmDetTargets &o) {
  typedef void (*ColKern)(const FfmColArgs);
  constexpr int E = 4;   // column entries in flight per warp
  const bool ada = o.gnP != nullptr;
  ColKern ck = nullptr;
  size_t warpSmem = ffm_cols_warp_smem(E);
  int64_t taskMul = 1;   // warp tasks per column segment
  if (tunedKernel && !ada) {
    ck = m->k == 4 ? ffm_cols_grad_kernel<4, E> : m->k == 8 ? ffm_cols_grad_kernel<8, E> : ffm_cols_grad_kernel<16, E>;
  } else if (tunedKernel) {
    // AdaGrad: at k = 16 two entries in flight leave room for the square accumulators (ptxas)
    ck = m->k == 4 ? ffm_cols_grad_kernel<4, E, true> : m->k == 8 ? ffm_cols_grad_kernel<8, E, true>
                                                                  : ffm_cols_grad_kernel<16, 2, true>;
    warpSmem = ffm_cols_warp_smem(m->k == 16 ? 2 : E);
  } else {
    const int kt = ada ? ffm_cols_ada_kt(m->k) : ffm_cols_generic_kt(m->k);
    int gE;
    if (!ada) {
      switch (kt) {   // entries per batch: the most without spills (ptxas), 24-64 partner components per lane in flight
        case 4: ck = ffm_cols_grad_generic_kernel<4, 6>; gE = 6; break;
        case 8: ck = ffm_cols_grad_generic_kernel<8, 4>; gE = 4; break;
        case 16: ck = ffm_cols_grad_generic_kernel<16, 4>; gE = 4; break;
        default: ck = ffm_cols_grad_generic_kernel<32, 2>; gE = 2; break;
      }
    } else {
      switch (kt) {   // the same entries per batch as the gradient's instances: still no spills (ptxas)
        case 4: ck = ffm_cols_grad_generic_kernel<4, 6, true>; gE = 6; break;
        case 8: ck = ffm_cols_grad_generic_kernel<8, 4, true>; gE = 4; break;
        default: ck = ffm_cols_grad_generic_kernel<16, 4, true>; gE = 4; break;
      }
    }
    warpSmem = ffm_cols_generic_warp_smem(gE);
    taskMul = (m->nFields + 31) / 32 * ((m->k + kt - 1) / kt);   // (segment, block of 32 fields, component chunk)
  }
  int rc;
  const int SB8 = (int)(m->nFields * m->k);
  const size_t slotLen = (size_t)(ada ? 2 : 1) * (SB8 + 1);
  const size_t need = (size_t)std::max<int64_t>(nRows, 1) + (size_t)tw->nSlots * slotLen + 16;
  if (ctx->stashCap < need) {
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->stash) CK(cudaFree(ctx->stash));
    ctx->stash = nullptr;
    ctx->stashCap = 0;
    if (cudaMalloc(&ctx->stash, need * 8) != cudaSuccess) {
      (void)cudaGetLastError();   // an allocation failure is not sticky: later calls must not see it
      ctx->stash = nullptr;
      return nimfm_fail(ctx, NIMFM_ERR_CUDA,
                        "the deterministic FFM gradient could not allocate its stash: %zu bytes = 8 x (nRows %lld + "
                        "%lld column partial sums x (nFields x nComponents %d + 1))",
                        need * 8, (long long)nRows, (long long)tw->nSlots, SB8);
    }
    ctx->stashCap = need;
  }
  // pass 1: the forward pair kernel leaves yhat per row, then coef = dloss / mb in place + the loss partials
  FfmPlan pl;
  if ((rc = ffm_plan_mode(ctx, m, X, nRows, FFM_PREDICT, &pl))) return rc;
  FfmArgs a;
  ffm_fill_args(a, m, X);
  a.b = o.b;
  a.rowBegin = rowBegin; a.nRows = nRows; a.yOut = ctx->stash; a.CH = pl.CH;
  pl.kern<<<pl.grid, pl.block, pl.smem, ctx->stream>>>(a);
  LAUNCHED(ctx);
  const int cgrid = (int)std::max<int64_t>(1, std::min<int64_t>((nRows + 255) / 256, (int64_t)ctx->numSMs * 4));
  if ((rc = nimfm_ensure_partials(ctx, (size_t)cgrid * 4))) return rc;
  dloss_coef_kernel<<<cgrid, 256, 0, ctx->stream>>>(ctx->stash, X->y, rowBegin, nRows, loss, thr, mb, ctx->partials);
  LAUNCHED(ctx);
  reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(ctx->partials, cgrid, o.red4, 0);
  LAUNCHED(ctx);
  // pass 2: the column kernel
  FfmColArgs c;
  memset(&c, 0, sizeof(c));
  c.cdata = tw->csc->data; c.crow = tw->csc->indices;
  c.taskCol = tw->taskCol; c.taskLen = tw->taskLen; c.taskSlot = tw->taskSlot; c.taskBeg = tw->taskBeg;
  c.nTasks = tw->nTasks;
  c.data = X->data; c.indices = X->indices; c.fields = X->fields; c.indptr = X->indptr;
  c.coef = ctx->stash;
  c.rowBegin = rowBegin; c.rowEnd = rowBegin + nRows;
  c.nFields = (int)m->nFields; c.CH = (int)std::max<int64_t>(X->maxSegNnz, 1);
  c.d = m->d;
  if (!m->PT) CK(cudaMalloc(&m->PT, (size_t)m->nP() * 8));
  ffm_field_major_kernel<<<ew_grid(ctx, m->nP()), 256, 0, ctx->stream>>>(m->P, m->PT, m->d, (int)m->nFields, m->k);
  LAUNCHED(ctx);
  c.PT = m->PT; c.gP = o.gP; c.gw = o.gw; c.gnP = o.gnP; c.gnw = o.gnw;
  c.partial = ctx->stash + std::max<int64_t>(nRows, 1);
  c.fitLinear = m->fitLinear;
  c.k = m->k;
  if (tw->nTasks > 0) {
    const int block = 128;   // 143 registers at k = 8: three 4-warp blocks per SM
    const size_t smem = (size_t)(block / 32) * warpSmem;
    CK(cudaFuncSetAttribute(ck, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int occ = 0;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ck, block, smem));
    if (!tunedKernel) occ = std::min(occ, FFM_COLS_GENERIC_BLOCKS_PER_SM);
    const int64_t wantBlocks = (tw->nTasks * taskMul + block / 32 - 1) / (block / 32);
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(wantBlocks, (int64_t)std::max(occ, 1) * ctx->numSMs));
    ck<<<grid, block, smem, ctx->stream>>>(c);
    LAUNCHED(ctx);
  }
  if (tw->nMulti > 0) {
    if (ada)
      ffm_cols_combine_ada_kernel<<<(unsigned)tw->nMulti, 128, 0, ctx->stream>>>(
          tw->multiCol, tw->multiFirst, tw->multiCount, tw->nMulti, c.partial, SB8, c.gP, c.gw, c.gnP, c.gnw,
          m->fitLinear);
    else
      ffm_cols_combine_kernel<<<(unsigned)tw->nMulti, 128, 0, ctx->stream>>>(tw->multiCol, tw->multiFirst,
                                                                             tw->multiCount, tw->nMulti, c.partial, SB8,
                                                                             c.gP, c.gw, m->fitLinear);
    LAUNCHED(ctx);
  }
  CK(cudaGetLastError());
  return NIMFM_OK;
}

// the tuned column kernel's shape limits (ffm_cols.cuh), and whether it runs: NIMFM_FFM_COLS=generic puts the generic
// kernel in its place
static bool ffm_cols_tuned_shape(const nimfm_ffm *m, const nimfm_dataset *X) {
  const int CH = (int)std::max<int64_t>(X->maxSegNnz, 1);
  return (m->k == 4 || m->k == 8 || m->k == 16) && CH <= 64 && m->nFields <= 64 &&
         m->d * m->nFields < (int64_t)2147483647;
}
static bool ffm_cols_want_generic() {
  const char *envC = getenv("NIMFM_FFM_COLS");
  return envC && !strcmp(envC, "generic");
}

// a column entry is a sample's whole gradient element only when its row holds one nonzero per field
static int ffm_det_require_one_per_field(nimfm_ctx *ctx, const nimfm_dataset *X) {
  bool dups = true;
  int rc;
  if ((rc = ffm_has_field_dups(ctx, X, &dups))) return rc;
  if (dups)
    return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "the deterministic FFM gradient needs rows with one nonzero per "
                      "field (a row of this dataset repeats a field)");
  return NIMFM_OK;
}

static int ffm_launch_grad_cols(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, int loss, double thr,
                                int64_t rowBegin, int64_t nRows, const int32_t *rowIdxDev, double mb) {
  if (rowIdxDev || rowBegin < 0 || rowBegin + nRows > X->n)
    return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED,
                      "the deterministic FFM gradient needs a contiguous row range (no row list, no wrap-around)");
  int rc;
  if ((rc = ffm_det_require_one_per_field(ctx, X))) return rc;
  nimfm_det_twin *tw = nullptr;
  if ((rc = nimfm_det_twin_get(ctx, X, 0, &tw))) return rc;
  const FfmDetTargets o{m->grad, m->grad + m->nP(), nullptr, nullptr, ctx->scalars + 8, m->b};
  return ffm_det_pass(ctx, m, X, tw, loss, thr, rowBegin, nRows, mb,
                      ffm_cols_tuned_shape(m, X) && !ffm_cols_want_generic(), o);
}

static int ffm_launch_grad(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, int loss, double thr,
                           int64_t rowBegin, int64_t nRows, const int32_t *rowIdxDev, double mb) {
  if (const char *env = getenv("NIMFM_DETERMINISTIC"); env && env[0] == '1' && nRows > 0)
    return ffm_launch_grad_cols(ctx, m, X, loss, thr, rowBegin, nRows, rowIdxDev, mb);
  FfmPlan pl;
  int rc = ffm_plan_mode(ctx, m, X, nRows, FFM_GRAD, &pl, (reinterpret_cast<uintptr_t>(m->grad) & 15) == 0);
  if (rc) return rc;
  if ((rc = nimfm_ensure_partials(ctx, (size_t)pl.partialRows * 4))) return rc;
  FfmArgs a;
  ffm_fill_args(a, m, X);
  a.rowBegin = rowBegin; a.nRows = nRows; a.rowIdx = rowIdxDev;
  a.gP = m->grad; a.gw = m->grad + m->nP(); a.partials = ctx->partials;
  a.loss = loss; a.thr = thr; a.mb = mb; a.CH = pl.CH;
  pl.kern<<<pl.grid, pl.block, pl.smem, ctx->stream>>>(a);
  LAUNCHED(ctx);
  reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(ctx->partials, pl.partialRows, ctx->scalars + 8, 0);
  LAUNCHED(ctx);
  return NIMFM_OK;
}

// the gradient of one minibatch of the minibatch-SGD epoch (rows rowIdxDev[0 .. nRows), or the cursor
// (rowBegin + q) mod n) into m->grad, red4 at ctx->scalars + 8, for sgd_mb.cu.  Under NIMFM_DETERMINISTIC=1 a row list
// or a cursor that wraps past the last row gets the minibatch's own column index (nimfm_mb_index_build) and the column
// route runs over its view (as in nimfm_fm_launch_grad_rows); every other minibatch takes ffm_launch_grad as before.
int nimfm_ffm_launch_grad_rows(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, int loss, double thr,
                               int64_t rowBegin, int64_t nRows, const int32_t *rowIdxDev, double mb) {
  const char *env = getenv("NIMFM_DETERMINISTIC");
  if (!(env && env[0] == '1') || (!rowIdxDev && rowBegin + nRows <= X->n))
    return ffm_launch_grad(ctx, m, X, loss, thr, rowBegin, nRows, rowIdxDev, mb);
  int rc;
  if ((rc = ffm_det_require_one_per_field(ctx, X))) return rc;
  nimfm_trace_begin(ctx, "det index");
  nimfm_mb_index *ix = nullptr;
  rc = nimfm_mb_index_build(ctx, X, 0, rowBegin, nRows, rowIdxDev, &ix);
  nimfm_trace_end(ctx);
  if (rc) return rc;
  nimfm_trace_begin(ctx, "det passes");
  const FfmDetTargets o{m->grad, m->grad + m->nP(), nullptr, nullptr, ctx->scalars + 8, m->b};
  rc = ffm_det_pass(ctx, m, &ix->view, &ix->tw, loss, thr, 0, nRows, mb,
                    ffm_cols_tuned_shape(m, X) && !ffm_cols_want_generic(), o);
  nimfm_trace_end(ctx);
  return rc;
}

int32_t nimfm_ffm_loss_grad(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, int32_t loss,
                            double huberThreshold, int64_t rowBegin, int64_t nRows, const int64_t *rowIdx,
                            int64_t miniBatchSize, int32_t zeroGrads, int32_t allreduce, double *lossSum) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int rc = check_ffm_ds(ctx, m, X, true);
  if (rc) return rc;
  REQUIRE(nRows >= 0 && miniBatchSize >= 1, "bad nRows / miniBatchSize");
  REQUIRE(rowIdx != nullptr || (rowBegin >= 0 && (rowBegin < X->n || nRows == 0)), "rowBegin out of range");
  const int64_t nG = m->nP() + m->d + 2;
  PeerScope peers(ctx, {allreduce ? m->grad : nullptr});
  if (peers.rc) return peers.rc;
  if (zeroGrads) CK(cudaMemsetAsync(m->grad, 0, (size_t)nG * 8, ctx->stream));
  const int32_t *idxDev = nullptr;
  if (rowIdx && nRows > 0) {
    if ((rc = nimfm_stage_row_ids(ctx, rowIdx, nRows, X->n))) return rc;
    idxDev = ctx->idx32Scratch;
  }
  if (nRows > 0) {
    if ((rc = ffm_launch_grad(ctx, m, X, loss, huberThreshold, rowBegin, nRows, idxDev, (double)miniBatchSize))) return rc;
    add_tail_kernel<<<1, 1, 0, ctx->stream>>>(m->grad + nG - 2, ctx->scalars + 8);
    LAUNCHED(ctx);
  }
  if (allreduce && (rc = nimfm_allreduce_sum(ctx, m->grad, nG))) return rc;
  CK(cudaGetLastError());
  if (lossSum) CK(cudaMemcpyAsync(lossSum, m->grad + nG - 1, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return NIMFM_OK;
}

int32_t nimfm_ffm_time_loss_grad(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, int32_t loss,
                                 int64_t nRows, int64_t miniBatchSize, int32_t reps, int32_t gradToo,
                                 float *msPerLaunch) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int rc = check_ffm_ds(ctx, m, X, gradToo != 0);
  if (rc) return rc;
  REQUIRE(reps >= 1 && nRows >= 1 && msPerLaunch, "bad arguments");
  FfmPlan pl;
  if ((rc = ffm_plan_mode(ctx, m, X, nRows, gradToo ? FFM_GRAD : FFM_PREDICT, &pl, (reinterpret_cast<uintptr_t>(m->grad) & 15) == 0)))
    return rc;
  FfmKernel kern = pl.kern;
  if ((rc = nimfm_ensure_partials(ctx, (size_t)pl.partialRows * 4))) return rc;
  double *dOut = nullptr;
  if (!gradToo) CK(cudaMalloc(&dOut, (size_t)nRows * 8));
  FfmArgs a;
  ffm_fill_args(a, m, X);
  a.nRows = nRows; a.yOut = dOut;
  a.gP = m->grad; a.gw = m->grad + m->nP(); a.partials = ctx->partials;
  a.loss = loss; a.thr = 1.0; a.mb = (double)miniBatchSize; a.CH = pl.CH;
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  for (int r = 0; r < reps; r++) {
    kern<<<pl.grid, pl.block, pl.smem, ctx->stream>>>(a);
    LAUNCHED(ctx);
  }
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  CK(cudaEventSynchronize(ctx->ev1));
  CK(cudaGetLastError());
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
  *msPerLaunch = ms / reps;
  if (dOut) CK(cudaFree(dOut));
  return NIMFM_OK;
}

// ------------------------------------------------------------------ AdaGrad for FFM (K11)
int32_t nimfm_ffm_adagrad_init(nimfm_ctx *ctx, nimfm_ffm *m, double eps, int32_t reset) {
  if (!ctx || !m) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  const int64_t nP = m->nP(), d = m->d;
  const bool fresh = !m->gsP;
  if (fresh) {
    CK(cudaMalloc(&m->gsP, (size_t)nP * 8));
    CK(cudaMalloc(&m->gnP, (size_t)nP * 8));
    CK(cudaMalloc(&m->gsw, (size_t)d * 8));
    CK(cudaMalloc(&m->gnw, (size_t)d * 8));
    { int rca = nimfm_comm_alloc(ctx, &m->dG, (size_t)(2 * nP + 3 * d + 8)); if (rca) return rca; }
    CK(cudaMalloc(&m->adaScal, 64));
  }
  if (fresh || reset) {
    CK(cudaMemsetAsync(m->gsP, 0, (size_t)nP * 8, ctx->stream));
    CK(cudaMemsetAsync(m->gsw, 0, (size_t)d * 8, ctx->stream));
    fill_kernel<<<ew_grid(ctx, nP), 256, 0, ctx->stream>>>(m->gnP, nP, eps);
    fill_kernel<<<ew_grid(ctx, d), 256, 0, ctx->stream>>>(m->gnw, d, eps);
    ctx->launches += 2;
    const double sc[2] = {0.0, eps};
    CK(cudaMemcpyAsync(m->adaScal, sc, 16, cudaMemcpyHostToDevice, ctx->stream));
  }
  CK(cudaMemsetAsync(m->dG, 0, (size_t)(2 * nP + 3 * d + 8) * 8, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  m->adaReady = true;
  return NIMFM_OK;
}

int32_t nimfm_ffm_adagrad_epoch(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_dataset *X, const nimfm_adagrad_cfg *cfg,
                                int64_t *it, const int64_t *perm, int64_t nRows, double *viol, double *lossSum) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  int rc = check_ffm_ds(ctx, m, X, true);
  if (rc) return rc;
  REQUIRE(cfg && it, "NULL argument");
  if (!m->adaReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_ffm_adagrad_init was not called");
  REQUIRE(cfg->miniBatchSize >= 1, "miniBatchSize < 1");
  REQUIRE(nRows >= 0 && (perm != nullptr || nRows <= X->n), "bad nRows");
  const int64_t nP = m->nP(), d = m->d;
  const int SB8 = (int)(m->nFields * m->k);
  const int32_t *idxDev = nullptr;
  if (perm && nRows > 0) {
    if ((rc = nimfm_stage_row_ids(ctx, perm, nRows, X->n))) return rc;
    idxDev = ctx->idx32Scratch;
  }
  CK(cudaMemsetAsync(ctx->scalars, 0, 16, ctx->stream));
  double *dGsP = m->dG, *dGnP = m->dG + nP, *dGsw = m->dG + 2 * nP, *dGnw = m->dG + 2 * nP + d;
  // delta block [dGsP | dGnP | dGsw | dGnw | loss, sum dL, sum dL^2, -], then per-feature row counts and
  // the refresh pass's viol (same scheme as nimfm_fm_adagrad_epoch)
  double *part = m->dG + 2 * nP + 2 * d;
  double *cntF = part + 4;
  double *violPart = cntF + d;
  const int64_t nDelta = 2 * nP + 2 * d + 4;
  const int64_t mb = cfg->miniBatchSize;
  MbSchedule sch;
  if ((rc = nimfm_mb_schedule(ctx, nRows, mb, *it, &sch))) return rc;
  PeerScope peers(ctx, {m->dG});
  if (peers.rc) return peers.rc;
  // NIMFM_DETERMINISTIC=1 with miniBatchSize > 1: the gradient sums and their squares come from the column route
  // (ffm_cols.cuh) over the minibatch's own column index (nimfm_mb_index_build), added in sample order without
  // atomics.  A one-row minibatch of a row with one nonzero per field adds each element once: the RED route is
  // already reproducible there and keeps it.
  const char *envDet = getenv("NIMFM_DETERMINISTIC");
  const bool det = envDet && envDet[0] == '1' && mb > 1;
  TraceReport traceReport{ctx, "deterministic adagrad epoch", det};
  if (det) {
    bool dups = true;
    if ((rc = ffm_has_field_dups(ctx, X, &dups))) return rc;
    if (dups)
      return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "the deterministic FFM AdaGrad needs rows with one nonzero per "
                        "field (a row of this dataset repeats a field)");
  }
  for (int64_t t = 0; t < sch.T; t++) {
    const int64_t start = std::min(t * mb, nRows);
    const int64_t cnt = sch.local(t);   // 0 once this rank's (shorter) shard is used up: it still joins the collectives
    const int32_t *rows = idxDev ? idxDev + start : nullptr;
    const double tIt = (double)(*it - 1);
    const int first = (*it == 1);
    {
      // per-feature row counts of the batch (all ranks): viol weights + the touched-feature set
      const int cgrid = (int)std::min<int64_t>((cnt * 32 + 255) / 256, (int64_t)ctx->numSMs * 16);
      adagrad_count_kernel<<<cgrid < 1 ? 1 : cgrid, 256, 0, ctx->stream>>>(X->indices, X->indptr, X->n, start, cnt, rows,
                                                                          d, 0, cntF, X->hotSlot, X->hotList, X->nHot);
      LAUNCHED(ctx);
      if ((rc = nimfm_allreduce_sum(ctx, cntF, d))) return rc;
    }
    if (!first) {
      // adagrad.update for FFM refreshes all nFields x k entries of every row feature (adagrad.nim:93-99)
      const int rgrid = ew_grid(ctx, nP);
      if ((rc = nimfm_ensure_partials(ctx, (size_t)rgrid * 4))) return rc;
      adagrad_refresh_kernel<<<rgrid, 256, 0, ctx->stream>>>(m->P, m->gsP, m->gnP, d, SB8, cntF, m->w, m->gsw, m->gnw, d,
                                                             m->fitLinear, cfg->eta0, tIt, cfg->alpha, cfg->beta,
                                                             ctx->partials);
      LAUNCHED(ctx);
      reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(ctx->partials, rgrid, violPart, 0);
      LAUNCHED(ctx);
    }
    // one rank: accumulate straight into g_sum / g_norm (see nimfm_fm_adagrad_epoch)
    const bool direct = ctx->nranks == 1;
    if (det) {
      nimfm_trace_begin(ctx, "det index");
      nimfm_mb_index *ix = nullptr;
      rc = nimfm_mb_index_build(ctx, X, 0, start, cnt, rows, &ix);
      nimfm_trace_end(ctx);
      if (rc) return rc;
      nimfm_trace_begin(ctx, "det passes");
      // the intercept every row of the minibatch sees (the AdaGrad kernels' prologue)
      adagrad_bias_kernel<<<1, 1, 0, ctx->stream>>>(ix->bias, m->b, m->adaScal, m->fitIntercept, first, cfg->eta0, tIt,
                                                    cfg->alpha0);
      LAUNCHED(ctx);
      const FfmDetTargets o{direct ? m->gsP : dGsP, direct ? m->gsw : dGsw, direct ? m->gnP : dGnP,
                            direct ? m->gnw : dGnw, part, ix->bias};
      rc = ffm_det_pass(ctx, m, &ix->view, &ix->tw, cfg->loss, cfg->huberThreshold, 0, cnt, 1.0,
                        ffm_cols_tuned_shape(m, X) && !ffm_cols_want_generic(), o);
      nimfm_trace_end(ctx);
      if (rc) return rc;
    } else {
      FfmPlan pl;
      const bool aligned = ((reinterpret_cast<uintptr_t>(direct ? m->gsP : dGsP) | reinterpret_cast<uintptr_t>(direct ? m->gnP : dGnP)) & 15) == 0;
      if ((rc = ffm_plan_mode(ctx, m, X, cnt, FFM_ADAGRAD, &pl, aligned))) return rc;
      if ((rc = nimfm_ensure_partials(ctx, (size_t)pl.partialRows * 4))) return rc;
      FfmArgs a;
      ffm_fill_args(a, m, X);
      a.rowBegin = start; a.nRows = cnt; a.rowIdx = rows;
      a.gP = direct ? m->gsP : dGsP; a.gw = direct ? m->gsw : dGsw;
      a.dGnP = direct ? m->gnP : dGnP; a.dGnw = direct ? m->gnw : dGnw;
      a.partials = ctx->partials;
      a.loss = cfg->loss; a.thr = cfg->huberThreshold;
      a.gsP = m->gsP; a.gnP = m->gnP; a.gsw = m->gsw; a.gnw = m->gnw; a.adaScal = m->adaScal;
      a.eta0 = cfg->eta0; a.tIt = tIt; a.alpha0 = cfg->alpha0; a.alpha = cfg->alpha; a.beta = cfg->beta;
      a.first = first;
      a.CH = pl.CH;
      pl.kern<<<pl.grid, pl.block, pl.smem, ctx->stream>>>(a);
      LAUNCHED(ctx);
      reduce_partials_kernel<<<1, 256, 0, ctx->stream>>>(ctx->partials, pl.partialRows, part, 0);
      LAUNCHED(ctx);
    }
    if ((rc = nimfm_allreduce_sum(ctx, m->dG, nDelta))) return rc;
    adagrad_scalar_kernel<<<1, 1, 0, ctx->stream>>>(m->b, m->adaScal, part, violPart, ctx->scalars, m->fitIntercept,
                                                    cfg->eta0, tIt, cfg->alpha0, first);
    LAUNCHED(ctx);
    if (direct) {
      CK(cudaMemsetAsync(cntF, 0, (size_t)d * 8, ctx->stream));
    } else {
      adagrad_apply_kernel<<<ew_grid(ctx, nP), 256, 0, ctx->stream>>>(m->gsP, m->gnP, dGsP, dGnP, nP, m->gsw, m->gnw,
                                                                     dGsw, dGnw, d, m->fitLinear, cntF, d);
      LAUNCHED(ctx);
    }
    *it += sch.global(t);
  }
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(ctx->hostScalars, ctx->scalars, 16, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (lossSum) *lossSum = ctx->hostScalars[0];
  if (viol) *viol = ctx->hostScalars[1];
  return NIMFM_OK;
}

int32_t nimfm_ffm_adagrad_finalize(nimfm_ctx *ctx, nimfm_ffm *m, const nimfm_adagrad_cfg *cfg, int64_t it) {
  if (!ctx || !m || !cfg) return NIMFM_ERR_INVALID;
  if (!m->adaReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_ffm_adagrad_init was not called");
  CK(cudaSetDevice(ctx->device));
  adagrad_finalize_kernel<<<ew_grid(ctx, m->nP()), 256, 0, ctx->stream>>>(
      m->P, m->gsP, m->gnP, m->nP(), m->w, m->gsw, m->gnw, m->d, m->fitLinear, m->b, m->adaScal, m->fitIntercept,
      cfg->eta0, (double)(it - 1), cfg->alpha0, cfg->alpha, cfg->beta);
  LAUNCHED(ctx);
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaGetLastError());
  return NIMFM_OK;
}

// g_sum / g_norm for warm starts (adagrad.nim:15-16, kept by init :47-62).  gsP / gnP cross in the reference layout
// P[field][j][s] and go through the same permutation as the parameters; the intercept's pair is adaScal[0..1].
int32_t nimfm_ffm_adagrad_get_state(nimfm_ctx *ctx, nimfm_ffm *m, double *gsP, double *gnP, double *gsw, double *gnw,
                                    double *gsb, double *gnb) {
  if (!ctx || !m) return NIMFM_ERR_INVALID;
  if (!m->adaReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_ffm_adagrad_init was not called");
  CK(cudaSetDevice(ctx->device));
  int rc;
  if (gsP && (rc = ffm_permute(ctx, m, gsP, m->gsP, 0))) return rc;
  if (gnP && (rc = ffm_permute(ctx, m, gnP, m->gnP, 0))) return rc;
  if (gsw) CK(cudaMemcpyAsync(gsw, m->gsw, (size_t)m->d * 8, cudaMemcpyDeviceToHost, ctx->stream));
  if (gnw) CK(cudaMemcpyAsync(gnw, m->gnw, (size_t)m->d * 8, cudaMemcpyDeviceToHost, ctx->stream));
  double sc[2];
  CK(cudaMemcpyAsync(sc, m->adaScal, 16, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (gsb) *gsb = sc[0];
  if (gnb) *gnb = sc[1];
  return NIMFM_OK;
}

int32_t nimfm_ffm_adagrad_set_state(nimfm_ctx *ctx, nimfm_ffm *m, const double *gsP, const double *gnP,
                                    const double *gsw, const double *gnw, double gsb, double gnb) {
  if (!ctx || !m) return NIMFM_ERR_INVALID;
  if (!m->adaReady) return nimfm_fail(ctx, NIMFM_ERR_STATE, "nimfm_ffm_adagrad_init was not called");
  REQUIRE(gsP && gnP && gsw && gnw, "NULL state array");
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = ffm_permute(ctx, m, const_cast<double *>(gsP), m->gsP, 1))) return rc;
  if ((rc = ffm_permute(ctx, m, const_cast<double *>(gnP), m->gnP, 1))) return rc;
  const double sc[2] = {gsb, gnb};
  CK(cudaMemcpyAsync(m->gsw, gsw, (size_t)m->d * 8, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(m->gnw, gnw, (size_t)m->d * 8, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(m->adaScal, sc, 16, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return NIMFM_OK;
}

}  // extern "C"
