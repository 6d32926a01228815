// dataset_ops.cu -- device-side integer bookkeeping on resident datasets (SURVEY a3, K12):
//   X[indicesRow]            tensor/sparse.nim:263-285  (CSR / CSR-with-fields row gather)
//   X[a..b] on a CSC         tensor/sparse.nim:300-325  (stable per-column filter, row ids rebased)
//   vstack                   tensor/sparse.nim:564-610  (CSR: concatenation; CSC: per-column interleave)
//   toCSCMatrix/toCSRMatrix  tensor/sparse.nim:490-527  (stable counting sort == stable radix sort by the
//                                                       other axis; within a column rows stay ascending)
// Everything here must be BIT-EXACT with the reference (same indptr, same within-segment order); the
// parity tests download the result and compare with the oracle's restatement.
// Scans / the radix sort come from CUB (ships with the CUDA toolkit); this is set-up work, not the hot path.
#include <cub/cub.cuh>

#include <algorithm>

#include "common.cuh"

namespace {

struct DsGuard {   // owns a dataset under construction: freed on every early return, released on success
  nimfm_ctx *ctx;
  nimfm_dataset *ds;
  DsGuard(nimfm_ctx *c, nimfm_dataset *d) : ctx(c), ds(d) {}
  ~DsGuard() { if (ds) nimfm_dataset_free(ctx, ds); }
  nimfm_dataset *release() { nimfm_dataset *d = ds; ds = nullptr; return d; }
};

struct DevBuf {   // frees on scope exit so early returns do not leak
  void *p = nullptr;
  ~DevBuf() { cudaFree(p); }
  template <class T> T *as() { return reinterpret_cast<T *>(p); }
};

__global__ void seg_len_kernel(const int64_t *indptr, const int64_t *rows, int64_t nIdx, int64_t *len) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nIdx; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = rows[q];
    len[q] = indptr[r + 1] - indptr[r];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) len[nIdx] = 0;
}

// one warp per output row: copy the source row's nonzeros
__global__ void gather_rows_kernel(const int64_t *srcPtr, const int64_t *dstPtr, const int64_t *rows, int64_t nIdx,
                                   const double *sData, const int32_t *sIdx, const int32_t *sFld, double *dData,
                                   int32_t *dIdx, int32_t *dFld, const double *sY, double *dY) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nWarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t q = warp; q < nIdx; q += nWarps) {
    const int64_t r = rows[q];
    const int64_t sb = srcPtr[r], db = dstPtr[q], z = srcPtr[r + 1] - sb;
    for (int64_t t = lane; t < z; t += 32) {
      dData[db + t] = sData[sb + t];
      dIdx[db + t] = sIdx[sb + t];
      if (sFld) dFld[db + t] = sFld[sb + t];
    }
    if (lane == 0 && sY) dY[q] = sY[r];
  }
}

__global__ void flag_range_kernel(const int32_t *idx, int64_t nnz, int32_t lo, int32_t hi, int64_t *flag) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q <= nnz; q += (int64_t)gridDim.x * blockDim.x)
    flag[q] = (q < nnz && idx[q] >= lo && idx[q] <= hi) ? 1 : 0;
}

__global__ void compact_range_kernel(const int32_t *idx, const double *data, int64_t nnz, int32_t lo, int32_t hi,
                                     const int64_t *pos, int32_t *oIdx, double *oData) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nnz; q += (int64_t)gridDim.x * blockDim.x) {
    const int32_t i = idx[q];
    if (i >= lo && i <= hi) {
      oIdx[pos[q]] = i - lo;
      oData[pos[q]] = data[q];
    }
  }
}

__global__ void remap_ptr_kernel(const int64_t *inPtr, int64_t nSeg, const int64_t *pos, int64_t *outPtr) {
  for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s <= nSeg; s += (int64_t)gridDim.x * blockDim.x)
    outPtr[s] = pos[inPtr[s]];
}

// out segment s = part segment s placed at outPtr[s] + off[s]; indices shifted by idxShift
__global__ void place_segments_kernel(const int64_t *pPtr, int64_t nSeg, const int64_t *outPtr, const int64_t *off,
                                      const double *pData, const int32_t *pIdx, const int32_t *pFld, int32_t idxShift,
                                      double *oData, int32_t *oIdx, int32_t *oFld) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nWarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t s = warp; s < nSeg; s += nWarps) {
    const int64_t sb = pPtr[s], z = pPtr[s + 1] - sb, db = outPtr[s] + (off ? off[s] : 0);
    for (int64_t t = lane; t < z; t += 32) {
      oData[db + t] = pData[sb + t];
      oIdx[db + t] = pIdx[sb + t] + idxShift;
      if (pFld) oFld[db + t] = pFld[sb + t];
    }
  }
}

__global__ void add_seg_len_kernel(const int64_t *pPtr, int64_t nSeg, int64_t *acc, int64_t *offBefore) {
  for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < nSeg; s += (int64_t)gridDim.x * blockDim.x) {
    if (offBefore) offBefore[s] = acc[s];
    acc[s] += pPtr[s + 1] - pPtr[s];
  }
}

__global__ void shift_ptr_kernel(const int64_t *pPtr, int64_t nSeg, int64_t base, int64_t *outPtr) {
  // outPtr[1 + s] = base + pPtr[1 + s]  (vstack of CSR: indptr &= X.indptr[1..^1].map(x => nnz + x))
  for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < nSeg; s += (int64_t)gridDim.x * blockDim.x)
    outPtr[1 + s] = base + pPtr[1 + s];
}

// expand indptr into one segment id per nonzero (warp per segment), and the identity permutation
__global__ void expand_seg_ids_kernel(const int64_t *ptr, int64_t nSeg, int32_t *segOf) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nWarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t s = warp; s < nSeg; s += nWarps)
    for (int64_t q = ptr[s] + lane; q < ptr[s + 1]; q += 32) segOf[q] = (int32_t)s;
}

__global__ void iota_kernel(uint32_t *p, int64_t n) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < n; q += (int64_t)gridDim.x * blockDim.x)
    p[q] = (uint32_t)q;
}

__global__ void permute_gather_kernel(const uint32_t *perm, int64_t nnz, const double *data, const int32_t *segOf,
                                      double *oData, int32_t *oIdx) {
  for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nnz; q += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t p = perm[q];
    oData[q] = data[p];
    oIdx[q] = segOf[p];
  }
}

// outPtr[t] = first position whose (sorted) key is >= t
__global__ void lower_bound_ptr_kernel(const int32_t *sortedKeys, int64_t nnz, int64_t nOut, int64_t *outPtr) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t <= nOut; t += (int64_t)gridDim.x * blockDim.x) {
    int64_t lo = 0, hi = nnz;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if ((int64_t)sortedKeys[mid] < t) lo = mid + 1; else hi = mid;
    }
    outPtr[t] = lo;
  }
}

__global__ void max_seg_kernel(const int64_t *ptr, int64_t nSeg, unsigned long long *out) {
  unsigned long long m = 0;
  for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < nSeg; s += (int64_t)gridDim.x * blockDim.x)
    m = max(m, (unsigned long long)(ptr[s + 1] - ptr[s]));
  for (int off = 16; off > 0; off >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, off));
  if ((threadIdx.x & 31) == 0 && m) atomicMax(out, m);
}

int grid_for(nimfm_ctx *ctx, int64_t items, int perBlock = 256) {
  int64_t g = (items + perBlock - 1) / perBlock;
  g = std::min<int64_t>(g, (int64_t)ctx->numSMs * 16);
  return (int)std::max<int64_t>(g, 1);
}

int exclusive_scan(nimfm_ctx *ctx, const int64_t *in, int64_t *out, int64_t n) {
  size_t tmpBytes = 0;
  CK(cub::DeviceScan::ExclusiveSum(nullptr, tmpBytes, in, out, n, ctx->stream));
  DevBuf tmp;
  CK(cudaMalloc(&tmp.p, tmpBytes ? tmpBytes : 16));
  CK(cub::DeviceScan::ExclusiveSum(tmp.p, tmpBytes, in, out, n, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return NIMFM_OK;
}

int finish_dataset(nimfm_ctx *ctx, nimfm_dataset *o, const nimfm_dataset *hotFrom) {
  const int64_t nSeg = o->kind == NIMFM_DS_CSC ? o->d : o->n;
  DevBuf m;
  CK(cudaMalloc(&m.p, 8));
  CK(cudaMemsetAsync(m.p, 0, 8, ctx->stream));
  if (nSeg > 0) {
    max_seg_kernel<<<grid_for(ctx, nSeg), 256, 0, ctx->stream>>>(o->indptr, nSeg, m.as<unsigned long long>());
    LAUNCHED(ctx);
  }
  unsigned long long h = 0;
  CK(cudaMemcpyAsync(&h, m.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  o->maxSegNnz = (int64_t)h;
  if (o->kind != NIMFM_DS_CSC) {
    // derived row sets keep the parent's hot-column table (bookkeeping only: it selects where the
    // gradients of those columns are accumulated, never what is computed)
    const size_t tab = (size_t)std::max<int64_t>(o->d, 1);
    CK(cudaMalloc(&o->hotSlot, tab));
    CK(cudaMalloc(&o->hotList, 16 * sizeof(int32_t)));
    if (hotFrom && hotFrom->hotSlot && hotFrom->d == o->d) {
      CK(cudaMemcpyAsync(o->hotSlot, hotFrom->hotSlot, tab, cudaMemcpyDeviceToDevice, ctx->stream));
      CK(cudaMemcpyAsync(o->hotList, hotFrom->hotList, 16 * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
      o->nHot = hotFrom->nHot;
    } else {
      CK(cudaMemsetAsync(o->hotSlot, 255, tab, ctx->stream));
      o->nHot = 0;
    }
    CK(cudaStreamSynchronize(ctx->stream));
  }
  CK(cudaGetLastError());
  return NIMFM_OK;
}

int alloc_arrays(nimfm_ctx *ctx, nimfm_dataset *o, int64_t nSeg, int64_t nnz, bool fields) {
  CK(cudaMalloc(&o->indptr, ((size_t)nSeg + 1) * 8));
  CK(cudaMalloc(&o->data, (size_t)std::max<int64_t>(nnz, 2) * 8));
  CK(cudaMalloc(&o->indices, (size_t)std::max<int64_t>(nnz, 4) * 4));
  if (fields) CK(cudaMalloc(&o->fields, (size_t)std::max<int64_t>(nnz, 4) * 4));
  return NIMFM_OK;
}

}  // namespace

// The stable sort at the core of nimfm_dataset_transpose: the nnz entries of nsIn input segments (inPtr, inIdx = the
// other axis, inData) sorted by inIdx with a stable radix sort, so entries of one output segment keep input order ->
// outData, outIdx (the input segment of each entry) and outPtr[0 .. nsOut].  All buffers are the caller's.  With
// s->tmp == nullptr it only sets s->tmpBytes, the CUB scratch the call needs, and launches nothing.
int nimfm_transpose_sort(nimfm_ctx *ctx, int64_t nsIn, int64_t nsOut, int64_t nnz, const int64_t *inPtr,
                         const int32_t *inIdx, const double *inData, TransposeScratch *s, double *outData,
                         int32_t *outIdx, int64_t *outPtr) {
  int endBit = 1;
  while (endBit < 31 && ((int64_t)1 << endBit) < nsOut) endBit++;
  if (!s->tmp) {
    s->tmpBytes = 0;
    if (nnz > 0)
      CK(cub::DeviceRadixSort::SortPairs(nullptr, s->tmpBytes, inIdx, s->keysOut, s->permIn, s->permOut, (int)nnz, 0,
                                         endBit, ctx->stream));
    return NIMFM_OK;
  }
  if (nnz > 0) {
    expand_seg_ids_kernel<<<grid_for(ctx, nsIn * 32), 256, 0, ctx->stream>>>(inPtr, nsIn, s->segOf);
    iota_kernel<<<grid_for(ctx, nnz), 256, 0, ctx->stream>>>(s->permIn, nnz);
    ctx->launches += 2;
    size_t tmpBytes = s->tmpBytes;
    CK(cub::DeviceRadixSort::SortPairs(s->tmp, tmpBytes, inIdx, s->keysOut, s->permIn, s->permOut, (int)nnz, 0, endBit,
                                       ctx->stream));
    permute_gather_kernel<<<grid_for(ctx, nnz), 256, 0, ctx->stream>>>(s->permOut, nnz, inData, s->segOf, outData,
                                                                      outIdx);
    LAUNCHED(ctx);
  }
  lower_bound_ptr_kernel<<<grid_for(ctx, nsOut + 1), 256, 0, ctx->stream>>>(s->keysOut, nnz, nsOut, outPtr);
  LAUNCHED(ctx);
  return NIMFM_OK;
}

// ------------------------------------------------------------------ the column index of one minibatch
// nimfm_mb_index_build (common.cuh).  Everything below runs on the stream; the host reads back four counts once.
namespace {

constexpr int MB_SEG = 512;   // entries per column segment: the SEG of the dataset twin (fm_cols.cu)

struct SegCount {   // per column: segments (tasks), 1 if the column has several, partial slots
  long long tasks, multi, slots;
};
struct SegCountSum {
  __host__ __device__ SegCount operator()(const SegCount &a, const SegCount &b) const {
    return {a.tasks + b.tasks, a.multi + b.multi, a.slots + b.slots};
  }
};

// one warp per minibatch position q: its source row (rowIdx[q], or (rowBegin + q) mod n: a cursor that wraps past the
// last row), its length, and the per-column entry counts (hot columns of the dataset are counted in shared memory
// first, as in adagrad_count_kernel, so they do not serialise on one counter)
__global__ void mb_rows_kernel(const int64_t *indptr, const int32_t *indices, int64_t n, int64_t rowBegin,
                               int64_t nRows, const int32_t *rowIdx, int64_t *rows, int64_t *len, int64_t *colCnt,
                               const uint8_t *hotSlot, const int32_t *hotList, int nHot) {
  __shared__ unsigned long long hotCnt[16];
  if (threadIdx.x < 16) hotCnt[threadIdx.x] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nWarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t q = warp; q < nRows; q += nWarps) {
    const int64_t r = rowIdx ? (int64_t)rowIdx[q] : (rowBegin + q) % n;
    if (lane == 0) {
      rows[q] = r;
      len[q] = indptr[r + 1] - indptr[r];
    }
    for (int64_t e = indptr[r] + lane; e < indptr[r + 1]; e += 32) {
      const int32_t j = indices[e];
      const int slot = (hotSlot && nHot > 0) ? hotSlot[j] : 255;
      if (slot != 255) atomicAdd(&hotCnt[slot], 1ull);
      else atomicAdd(reinterpret_cast<unsigned long long *>(colCnt + j), 1ull);
    }
  }
  if (warp == 0 && lane == 0) len[nRows] = 0;
  __syncthreads();
  if ((int)threadIdx.x < nHot && hotCnt[threadIdx.x] > 0)
    atomicAdd(reinterpret_cast<unsigned long long *>(colCnt + hotList[threadIdx.x]), hotCnt[threadIdx.x]);
}

// per column j < d + nAug (dummy columns d + a hold every position): its segment counts; entry d + nAug is zero so
// that the exclusive scan ends with the totals
__global__ void mb_seg_count_kernel(const int64_t *colCnt, int64_t d, int nAug, int64_t nRows, SegCount *out) {
  const int64_t dd = d + nAug;
  for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j <= dd; j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t L = j < d ? colCnt[j] : (j < dd ? nRows : 0);
    const long long nseg = (L + MB_SEG - 1) / MB_SEG;
    out[j] = {nseg, nseg > 1 ? 1 : 0, nseg > 1 ? nseg : 0};
  }
}

__global__ void mb_totals_kernel(const int64_t *viewPtr, int64_t nRows, const SegCount *off, int64_t dd, int64_t *tot) {
  tot[0] = viewPtr[nRows];
  tot[1] = off[dd].tasks;
  tot[2] = off[dd].multi;
  tot[3] = off[dd].slots;
}

// the segment table in the dataset twin's layout (build_twin, fm_cols.cu), one thread per column
__global__ void mb_seg_table_kernel(const int64_t *colPtr, int64_t d, int nAug, int64_t nRows, const SegCount *off,
                                    int32_t *taskCol, int64_t *taskBeg, int32_t *taskLen, int32_t *taskSlot,
                                    int32_t *multiCol, int32_t *multiFirst, int32_t *multiCount) {
  const int64_t dd = d + nAug;
  for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < dd; j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = j < d ? colPtr[j] : 0, e = j < d ? colPtr[j + 1] : nRows;
    const SegCount o = off[j];
    const int64_t nseg = (e - b + MB_SEG - 1) / MB_SEG;
    if (nseg > 1) {
      multiCol[o.multi] = (int32_t)j;
      multiFirst[o.multi] = (int32_t)o.slots;
      multiCount[o.multi] = (int32_t)nseg;
    }
    for (int64_t s = 0; s < nseg; s++) {
      const int64_t t = o.tasks + s;
      taskCol[t] = (int32_t)j;
      taskBeg[t] = b + s * MB_SEG;
      const int64_t left = e - (b + s * MB_SEG);
      taskLen[t] = (int32_t)(left < MB_SEG ? left : MB_SEG);
      taskSlot[t] = nseg > 1 ? (int32_t)(o.slots + s) : -1;
    }
  }
}

// grow *p to hold n elements of T (contents are not kept)
template <class T>
int grow(nimfm_ctx *ctx, T **p, size_t &cap, size_t n) {
  if (n <= cap && *p) return NIMFM_OK;
  n = std::max<size_t>(n + n / 4, 16);
  CK(cudaFree(*p));
  *p = nullptr;
  cap = 0;
  if (cudaMalloc(p, n * sizeof(T)) != cudaSuccess) {
    (void)cudaGetLastError();   // not sticky: the caller reports it
    *p = nullptr;
    return nimfm_fail(ctx, NIMFM_ERR_CUDA, "the minibatch column index could not allocate %zu bytes", n * sizeof(T));
  }
  cap = n;
  return NIMFM_OK;
}

}  // namespace

void nimfm_mb_index_free(nimfm_mb_index *m) {
  if (!m) return;
  void *bufs[] = {m->rows, m->rowLen, m->ptr, m->data, m->idx, m->fld, m->y, m->cPtr, m->cData, m->cIdx, m->segOf,
                  m->keysOut, m->permIn, m->permOut, m->tmp, m->colCnt, m->segOff, m->taskCol, m->taskBeg, m->taskLen,
                  m->taskSlot, m->multiCol, m->multiFirst, m->multiCount, m->tot, m->bias, m->yhat};
  for (void *p : bufs) cudaFree(p);
  cudaFreeHost(m->hostTot);
  delete m;
}

int nimfm_mb_index_build(nimfm_ctx *ctx, const nimfm_dataset *X, int nAug, int64_t rowBegin, int64_t nRows,
                         const int32_t *rowIdx, nimfm_mb_index **out) {
  REQUIRE(X->kind == NIMFM_DS_CSR || X->kind == NIMFM_DS_CSR_FIELD, "the minibatch column index needs a CSR dataset");
  REQUIRE(nRows >= 0 && (rowIdx || (rowBegin >= 0 && (rowBegin < X->n || rowBegin + nRows <= X->n))),
          "bad minibatch rows");
  if (!ctx->mbIndex) ctx->mbIndex = new nimfm_mb_index();
  nimfm_mb_index *m = ctx->mbIndex;
  const int64_t d = X->d, dd = d + nAug, B = nRows;
  int rc;
  // 1. rows, lengths and column counts of the minibatch; its indptr and the segment counts by two scans
  if ((rc = grow(ctx, &m->rows, m->capRows, (size_t)B + 1)) || (rc = grow(ctx, &m->rowLen, m->capRowLen, (size_t)B + 1)) ||
      (rc = grow(ctx, &m->ptr, m->capPtr, (size_t)B + 1)) || (rc = grow(ctx, &m->y, m->capY, (size_t)B + 1)) ||
      (rc = grow(ctx, &m->colCnt, m->capCol, (size_t)d + 1)) || (rc = grow(ctx, &m->cPtr, m->capColPtr, (size_t)d + 1)) ||
      (rc = grow(ctx, &m->segOff, m->capSeg, 6 * ((size_t)dd + 1))) || (rc = grow(ctx, &m->tot, m->capTot, 4)) ||
      (rc = grow(ctx, &m->bias, m->capBias, 1)) || (rc = grow(ctx, &m->yhat, m->capYhat, (size_t)B + 1)))
    return rc;
  if (!m->hostTot) CK(cudaMallocHost(&m->hostTot, 4 * sizeof(int64_t)));
  SegCount *cnt = reinterpret_cast<SegCount *>(m->segOff), *off = cnt + dd + 1;
  CK(cudaMemsetAsync(m->colCnt, 0, (size_t)d * 8, ctx->stream));
  mb_rows_kernel<<<grid_for(ctx, B * 32), 256, 0, ctx->stream>>>(X->indptr, X->indices, X->n, rowBegin, B, rowIdx,
                                                                m->rows, m->rowLen, m->colCnt, X->hotSlot, X->hotList,
                                                                X->nHot);
  LAUNCHED(ctx);
  mb_seg_count_kernel<<<grid_for(ctx, dd + 1), 256, 0, ctx->stream>>>(m->colCnt, d, nAug, B, cnt);
  LAUNCHED(ctx);
  size_t scanRows = 0, scanSeg = 0;
  CK(cub::DeviceScan::ExclusiveSum(nullptr, scanRows, m->rowLen, m->ptr, B + 1, ctx->stream));
  CK(cub::DeviceScan::ExclusiveScan(nullptr, scanSeg, cnt, off, SegCountSum(), SegCount{0, 0, 0}, dd + 1, ctx->stream));
  if ((rc = grow(ctx, &m->tmp, m->capTmp, std::max(scanRows, scanSeg)))) return rc;
  size_t tb = m->capTmp;
  CK(cub::DeviceScan::ExclusiveSum(m->tmp, tb, m->rowLen, m->ptr, B + 1, ctx->stream));
  tb = m->capTmp;
  CK(cub::DeviceScan::ExclusiveScan(m->tmp, tb, cnt, off, SegCountSum(), SegCount{0, 0, 0}, dd + 1, ctx->stream));
  mb_totals_kernel<<<1, 1, 0, ctx->stream>>>(m->ptr, B, off, dd, m->tot);
  LAUNCHED(ctx);
  // the one device-to-host copy of the minibatch: the entry count and the segment-table sizes
  CK(cudaMemcpyAsync(m->hostTot, m->tot, 4 * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  const int64_t nnz = m->hostTot[0], nTasks = m->hostTot[1], nMulti = m->hostTot[2], nSlots = m->hostTot[3];
  if (nnz > (int64_t)2147483647)
    return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED,
                      "a minibatch of %lld rows holds %lld nonzeros; the minibatch column index sorts with 32-bit "
                      "values and takes at most 2147483647 (use a smaller miniBatchSize)",
                      (long long)B, (long long)nnz);
  if (nSlots > (int64_t)2147483647)
    return nimfm_fail(ctx, NIMFM_ERR_UNSUPPORTED, "too many column segments in one minibatch (%lld)", (long long)nSlots);
  // 2. the gathered rows (the view) and their stable column-major twin
  const size_t e = (size_t)nnz + 1;
  if ((rc = grow(ctx, &m->data, m->capData, e)) || (rc = grow(ctx, &m->idx, m->capIdx, e)) ||
      (rc = grow(ctx, &m->cData, m->capCData, e)) || (rc = grow(ctx, &m->cIdx, m->capCIdx, e)) ||
      (rc = grow(ctx, &m->segOf, m->capSegOf, e)) || (rc = grow(ctx, &m->keysOut, m->capKeys, e)) ||
      (rc = grow(ctx, &m->permIn, m->capPermIn, e)) || (rc = grow(ctx, &m->permOut, m->capPermOut, e)) ||
      (X->fields && (rc = grow(ctx, &m->fld, m->capFld, e))) ||
      (rc = grow(ctx, &m->taskCol, m->capTaskCol, (size_t)nTasks + 1)) ||
      (rc = grow(ctx, &m->taskBeg, m->capTaskBeg, (size_t)nTasks + 1)) ||
      (rc = grow(ctx, &m->taskLen, m->capTaskLen, (size_t)nTasks + 1)) ||
      (rc = grow(ctx, &m->taskSlot, m->capTaskSlot, (size_t)nTasks + 1)) ||
      (rc = grow(ctx, &m->multiCol, m->capMultiCol, (size_t)nMulti + 1)) ||
      (rc = grow(ctx, &m->multiFirst, m->capMultiFirst, (size_t)nMulti + 1)) ||
      (rc = grow(ctx, &m->multiCount, m->capMultiCount, (size_t)nMulti + 1)))
    return rc;
  if (B > 0) {
    gather_rows_kernel<<<grid_for(ctx, B * 32), 256, 0, ctx->stream>>>(
        X->indptr, m->ptr, m->rows, B, X->data, X->indices, X->fields, m->data, m->idx, m->fld, X->y, m->y);
    LAUNCHED(ctx);
  }
  TransposeScratch s{m->segOf, m->keysOut, m->permIn, m->permOut, nullptr, 0};
  if ((rc = nimfm_transpose_sort(ctx, B, d, nnz, m->ptr, m->idx, m->data, &s, m->cData, m->cIdx, m->cPtr)))
    return rc;
  if ((rc = grow(ctx, &m->tmp, m->capTmp, s.tmpBytes))) return rc;
  s.tmp = m->tmp;
  s.tmpBytes = m->capTmp;
  if ((rc = nimfm_transpose_sort(ctx, B, d, nnz, m->ptr, m->idx, m->data, &s, m->cData, m->cIdx, m->cPtr)))
    return rc;
  // 3. the segment table
  if (dd > 0) {
    mb_seg_table_kernel<<<grid_for(ctx, dd), 256, 0, ctx->stream>>>(m->cPtr, d, nAug, B, off, m->taskCol, m->taskBeg,
                                                                    m->taskLen, m->taskSlot, m->multiCol, m->multiFirst,
                                                                    m->multiCount);
    LAUNCHED(ctx);
  }
  CK(cudaGetLastError());
  // the view keeps the parent's shape and planning facts (maxSegNnz picks the same row kernels), hot table and
  // field-repeat flag; the view, the twin and the table only point into the buffers above
  nimfm_dataset &v = m->view;
  v.kind = X->kind; v.n = B; v.d = d; v.nnz = nnz; v.nFields = X->nFields; v.maxSegNnz = X->maxSegNnz;
  v.data = m->data; v.indices = m->idx; v.indptr = m->ptr; v.fields = X->fields ? m->fld : nullptr;
  v.y = X->y ? m->y : nullptr;
  v.hotSlot = X->hotSlot; v.hotList = X->hotList; v.nHot = X->nHot; v.fieldDup = X->fieldDup;
  nimfm_dataset &c = m->csc;
  c.kind = NIMFM_DS_CSC; c.n = B; c.d = d; c.nnz = nnz;
  c.data = m->cData; c.indices = m->cIdx; c.indptr = m->cPtr;
  nimfm_det_twin &t = m->tw;
  t.csc = &m->csc;
  t.taskCol = m->taskCol; t.taskBeg = m->taskBeg; t.taskLen = m->taskLen; t.taskSlot = m->taskSlot;
  t.multiCol = m->multiCol; t.multiFirst = m->multiFirst; t.multiCount = m->multiCount;
  t.nTasks = nTasks; t.nMulti = nMulti; t.nSlots = nSlots; t.nAug = nAug;
  *out = m;
  return NIMFM_OK;
}

extern "C" {

// X[indicesRow] for CSRDataset / CSRFieldDataset (dataset.nim:319-367 -> tensor/sparse.nim:263-285);
// targets, when set, are gathered alongside (== shuffle(X, y, indices), dataset.nim:372-381).
int32_t nimfm_dataset_take_rows(nimfm_ctx *ctx, const nimfm_dataset *in, const int64_t *rowIdx, int64_t nIdx,
                                nimfm_dataset **out) {
  if (!ctx || !in) return NIMFM_ERR_INVALID;
  REQUIRE(out != nullptr, "out is NULL");
  REQUIRE(in->kind != NIMFM_DS_CSC, "Accessing row vectors by an index array is not supported for CSC");  // sparse.nim:298-299
  REQUIRE(nIdx >= 0 && (rowIdx != nullptr || nIdx == 0), "rowIdx is NULL");
  for (int64_t q = 0; q < nIdx; q++) {   // checkIndicesRow (sparse.nim:254-260)
    REQUIRE(rowIdx[q] < in->n, "max(indicesRow) %lld >= %lld.", (long long)rowIdx[q], (long long)in->n);
    REQUIRE(rowIdx[q] >= 0, "min(indicesRow) %lld < 0.", (long long)rowIdx[q]);
  }
  CK(cudaSetDevice(ctx->device));
  DevBuf rows, len;
  CK(cudaMalloc(&rows.p, (size_t)std::max<int64_t>(nIdx, 1) * 8));
  CK(cudaMalloc(&len.p, ((size_t)nIdx + 1) * 8));
  if (nIdx) CK(cudaMemcpyAsync(rows.p, rowIdx, (size_t)nIdx * 8, cudaMemcpyHostToDevice, ctx->stream));
  nimfm_dataset *o = new nimfm_dataset();
  DsGuard guard(ctx, o);
  o->kind = in->kind; o->n = nIdx; o->d = in->d; o->nFields = in->nFields;
  CK(cudaMalloc(&o->indptr, ((size_t)nIdx + 1) * 8));
  seg_len_kernel<<<grid_for(ctx, nIdx), 256, 0, ctx->stream>>>(in->indptr, rows.as<int64_t>(), nIdx, len.as<int64_t>());
  LAUNCHED(ctx);
  int rc = exclusive_scan(ctx, len.as<int64_t>(), o->indptr, nIdx + 1);
  if (rc) return rc;
  int64_t nnz = 0;
  CK(cudaMemcpy(&nnz, o->indptr + nIdx, 8, cudaMemcpyDeviceToHost));
  o->nnz = nnz;
  CK(cudaMalloc(&o->data, (size_t)std::max<int64_t>(nnz, 2) * 8));
  CK(cudaMalloc(&o->indices, (size_t)std::max<int64_t>(nnz, 4) * 4));
  if (in->fields) CK(cudaMalloc(&o->fields, (size_t)std::max<int64_t>(nnz, 4) * 4));
  if (in->y) CK(cudaMalloc(&o->y, (size_t)std::max<int64_t>(nIdx, 1) * 8));
  if (nIdx) {
    gather_rows_kernel<<<grid_for(ctx, nIdx * 32), 256, 0, ctx->stream>>>(
        in->indptr, o->indptr, rows.as<int64_t>(), nIdx, in->data, in->indices, in->fields, o->data, o->indices,
        o->fields, in->y, o->y);
    LAUNCHED(ctx);
  }
  if ((rc = finish_dataset(ctx, o, in))) return rc;
  *out = guard.release();
  return NIMFM_OK;
}

// X[first..last] (inclusive, as Nim's Slice).  CSR kinds: == X[toSeq(slice)] (sparse.nim:288-290);
// CSC: the O(nnz) per-column filter of sparse.nim:300-325 (entries keep their order, row ids -= first).
int32_t nimfm_dataset_slice_rows(nimfm_ctx *ctx, const nimfm_dataset *in, int64_t first, int64_t last,
                                 nimfm_dataset **out) {
  if (!ctx || !in) return NIMFM_ERR_INVALID;
  REQUIRE(out != nullptr, "out is NULL");
  REQUIRE(first >= 0, "min(indicesRow) %lld < 0.", (long long)first);
  REQUIRE(last < in->n, "max(indicesRow) %lld >= %lld.", (long long)last, (long long)in->n);
  REQUIRE(first <= last, "empty slice [%lld..%lld]", (long long)first, (long long)last);
  if (in->kind != NIMFM_DS_CSC) {
    std::vector<int64_t> ids((size_t)(last - first + 1));
    for (size_t q = 0; q < ids.size(); q++) ids[q] = first + (int64_t)q;
    return nimfm_dataset_take_rows(ctx, in, ids.data(), (int64_t)ids.size(), out);
  }
  CK(cudaSetDevice(ctx->device));
  const int64_t nnzIn = in->nnz, d = in->d;
  DevBuf flag, pos;
  CK(cudaMalloc(&flag.p, ((size_t)nnzIn + 1) * 8));
  CK(cudaMalloc(&pos.p, ((size_t)nnzIn + 1) * 8));
  flag_range_kernel<<<grid_for(ctx, nnzIn + 1), 256, 0, ctx->stream>>>(in->indices, nnzIn, (int32_t)first, (int32_t)last,
                                                                      flag.as<int64_t>());
  LAUNCHED(ctx);
  int rc = exclusive_scan(ctx, flag.as<int64_t>(), pos.as<int64_t>(), nnzIn + 1);
  if (rc) return rc;
  int64_t nnz = 0;
  CK(cudaMemcpy(&nnz, pos.as<int64_t>() + nnzIn, 8, cudaMemcpyDeviceToHost));
  nimfm_dataset *o = new nimfm_dataset();
  DsGuard guard(ctx, o);
  o->kind = NIMFM_DS_CSC; o->n = last - first + 1; o->d = d; o->nnz = nnz;
  if ((rc = alloc_arrays(ctx, o, d, nnz, false))) return rc;
  remap_ptr_kernel<<<grid_for(ctx, d + 1), 256, 0, ctx->stream>>>(in->indptr, d, pos.as<int64_t>(), o->indptr);
  LAUNCHED(ctx);
  if (nnzIn) {
    compact_range_kernel<<<grid_for(ctx, nnzIn), 256, 0, ctx->stream>>>(in->indices, in->data, nnzIn, (int32_t)first,
                                                                       (int32_t)last, pos.as<int64_t>(), o->indices,
                                                                       o->data);
    LAUNCHED(ctx);
  }
  if (in->y) {
    CK(cudaMalloc(&o->y, (size_t)o->n * 8));
    CK(cudaMemcpyAsync(o->y, in->y + first, (size_t)o->n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  }
  if ((rc = finish_dataset(ctx, o, nullptr))) return rc;
  *out = guard.release();
  return NIMFM_OK;
}

// vstack (dataset.nim:452-483 -> tensor/sparse.nim:564-640).  All parts of one kind and nFeatures.
int32_t nimfm_dataset_vstack(nimfm_ctx *ctx, const nimfm_dataset *const *parts, int32_t nParts, nimfm_dataset **out) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(out != nullptr && parts != nullptr && nParts >= 1, "bad arguments");
  const nimfm_dataset *p0 = parts[0];
  REQUIRE(p0 != nullptr, "NULL part");
  int64_t n = 0, nnz = 0;
  bool haveY = true;
  for (int i = 0; i < nParts; i++) {
    REQUIRE(parts[i] != nullptr, "NULL part");
    REQUIRE(parts[i]->kind == p0->kind, "all parts must be of one dataset kind");
    REQUIRE(parts[i]->d == p0->d, "All matrics must have the same shape[1].");   // sparse.nim:576-577
    REQUIRE(parts[i]->nFields == p0->nFields, "all parts must have the same nFields");
    n += parts[i]->n;
    nnz += parts[i]->nnz;
    haveY = haveY && (parts[i]->y != nullptr || parts[i]->n == 0);
  }
  REQUIRE(n < (int64_t)2147483647, "stacked row count does not fit int32");
  CK(cudaSetDevice(ctx->device));
  nimfm_dataset *o = new nimfm_dataset();
  DsGuard guard(ctx, o);
  o->kind = p0->kind; o->n = n; o->d = p0->d; o->nnz = nnz; o->nFields = p0->nFields;
  const bool csc = p0->kind == NIMFM_DS_CSC;
  const int64_t nSeg = csc ? o->d : n;
  int rc = alloc_arrays(ctx, o, nSeg, nnz, p0->fields != nullptr);
  if (rc) return rc;
  if (haveY && n > 0) CK(cudaMalloc(&o->y, (size_t)n * 8));
  if (!csc) {
    CK(cudaMemsetAsync(o->indptr, 0, 8, ctx->stream));
    int64_t rowBase = 0, nnzBase = 0;
    for (int i = 0; i < nParts; i++) {
      const nimfm_dataset *p = parts[i];
      if (p->n) {
        shift_ptr_kernel<<<grid_for(ctx, p->n), 256, 0, ctx->stream>>>(p->indptr, p->n, nnzBase, o->indptr + rowBase);
        LAUNCHED(ctx);
      }
      if (p->nnz) {
        CK(cudaMemcpyAsync(o->data + nnzBase, p->data, (size_t)p->nnz * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        CK(cudaMemcpyAsync(o->indices + nnzBase, p->indices, (size_t)p->nnz * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        if (p->fields)
          CK(cudaMemcpyAsync(o->fields + nnzBase, p->fields, (size_t)p->nnz * 4, cudaMemcpyDeviceToDevice, ctx->stream));
      }
      if (o->y && p->n) CK(cudaMemcpyAsync(o->y + rowBase, p->y, (size_t)p->n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
      rowBase += p->n;
      nnzBase += p->nnz;
    }
  } else {
    // column j of the result = column j of part 0, then of part 1 (row ids + n_0), ... (sparse.nim:598-609)
    const int64_t d = o->d;
    DevBuf acc, offs;
    CK(cudaMalloc(&acc.p, ((size_t)d + 1) * 8));
    CK(cudaMalloc(&offs.p, (size_t)std::max<int64_t>(d, 1) * 8 * nParts));
    CK(cudaMemsetAsync(acc.p, 0, ((size_t)d + 1) * 8, ctx->stream));
    for (int i = 0; i < nParts && d > 0; i++) {
      add_seg_len_kernel<<<grid_for(ctx, d), 256, 0, ctx->stream>>>(parts[i]->indptr, d, acc.as<int64_t>(),
                                                                   offs.as<int64_t>() + (size_t)i * d);
      LAUNCHED(ctx);
    }
    if ((rc = exclusive_scan(ctx, acc.as<int64_t>(), o->indptr, d + 1))) return rc;
    int64_t rowBase = 0;
    for (int i = 0; i < nParts; i++) {
      const nimfm_dataset *p = parts[i];
      if (d > 0 && p->nnz) {
        place_segments_kernel<<<grid_for(ctx, d * 32), 256, 0, ctx->stream>>>(
            p->indptr, d, o->indptr, offs.as<int64_t>() + (size_t)i * d, p->data, p->indices, nullptr, (int32_t)rowBase,
            o->data, o->indices, nullptr);
        LAUNCHED(ctx);
      }
      if (o->y && p->n) CK(cudaMemcpyAsync(o->y + rowBase, p->y, (size_t)p->n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
      rowBase += p->n;
    }
    CK(cudaStreamSynchronize(ctx->stream));
  }
  if ((rc = finish_dataset(ctx, o, p0))) return rc;
  *out = guard.release();
  return NIMFM_OK;
}

// toCSCMatrix / toCSRMatrix (tensor/sparse.nim:490-527) on the device: a STABLE radix sort of the
// nonzeros by their index along the other axis reproduces the reference's counting sort exactly
// (entries of one output segment stay in input-segment order).
int32_t nimfm_dataset_transpose(nimfm_ctx *ctx, const nimfm_dataset *in, nimfm_dataset **out) {
  if (!ctx || !in) return NIMFM_ERR_INVALID;
  REQUIRE(out != nullptr, "out is NULL");
  REQUIRE(in->kind != NIMFM_DS_CSR_FIELD, "transpose of field datasets is not supported");
  REQUIRE(in->nnz < (int64_t)2147483647, "nnz does not fit the 32-bit permutation");
  CK(cudaSetDevice(ctx->device));
  const bool toCsc = in->kind == NIMFM_DS_CSR;
  const int64_t nsIn = toCsc ? in->n : in->d, nsOut = toCsc ? in->d : in->n, nnz = in->nnz;
  nimfm_dataset *o = new nimfm_dataset();
  DsGuard guard(ctx, o);
  o->kind = toCsc ? NIMFM_DS_CSC : NIMFM_DS_CSR;
  o->n = in->n; o->d = in->d; o->nnz = nnz;
  int rc = alloc_arrays(ctx, o, nsOut, nnz, false);
  if (rc) return rc;
  DevBuf segOf, keysOut, permIn, permOut, tmp;
  const size_t n4 = (size_t)std::max<int64_t>(nnz, 4) * 4;
  CK(cudaMalloc(&segOf.p, n4));
  CK(cudaMalloc(&keysOut.p, n4));
  CK(cudaMalloc(&permIn.p, n4));
  CK(cudaMalloc(&permOut.p, n4));
  TransposeScratch s{segOf.as<int32_t>(), keysOut.as<int32_t>(), permIn.as<uint32_t>(), permOut.as<uint32_t>(), nullptr, 0};
  if ((rc = nimfm_transpose_sort(ctx, nsIn, nsOut, nnz, in->indptr, in->indices, in->data, &s, o->data, o->indices,
                                 o->indptr)))
    return rc;
  CK(cudaMalloc(&tmp.p, s.tmpBytes ? s.tmpBytes : 16));
  s.tmp = tmp.p;
  if ((rc = nimfm_transpose_sort(ctx, nsIn, nsOut, nnz, in->indptr, in->indices, in->data, &s, o->data, o->indices,
                                 o->indptr)))
    return rc;
  if (in->y) {
    CK(cudaMalloc(&o->y, (size_t)std::max<int64_t>(o->n, 1) * 8));
    CK(cudaMemcpyAsync(o->y, in->y, (size_t)o->n * 8, cudaMemcpyDeviceToDevice, ctx->stream));
  }
  CK(cudaStreamSynchronize(ctx->stream));
  if ((rc = finish_dataset(ctx, o, nullptr))) return rc;
  if (o->kind == NIMFM_DS_CSR && nnz > 0) {
    // a CSR made on the device has no host copy to sample: find the hot columns from the CSC side
    // (column length >= n/16), the 16 longest
    std::vector<int64_t> ptr((size_t)in->d + 1);
    CK(cudaMemcpy(ptr.data(), in->indptr, ((size_t)in->d + 1) * 8, cudaMemcpyDeviceToHost));
    std::vector<std::pair<int64_t, int64_t>> cand;
    for (int64_t j = 0; j < in->d; j++) {
      const int64_t len = ptr[j + 1] - ptr[j];
      if (len * 16 >= in->n && len >= 2) cand.push_back({len, j});
    }
    std::sort(cand.begin(), cand.end(), [](const std::pair<int64_t, int64_t> &x, const std::pair<int64_t, int64_t> &y) {
      return x.first != y.first ? x.first > y.first : x.second < y.second;
    });
    std::vector<int32_t> hot;
    for (size_t i = 0; i < cand.size() && i < 16; i++) hot.push_back((int32_t)cand[i].second);
    o->nHot = (int)hot.size();
    if ((rc = nimfm_upload_hot(ctx, hot, o->d, &o->hotSlot, &o->hotList))) return rc;
  }
  *out = guard.release();
  return NIMFM_OK;
}

}  // extern "C"
