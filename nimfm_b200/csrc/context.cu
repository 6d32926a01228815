// context.cu -- lifecycle, error plumbing, scratch pools, NCCL communicator (dlopen'ed lazily so the
// library loads on a box without NCCL/GPU; there is still no CPU compute path).
#include <dlfcn.h>
#include <stdarg.h>

#include <algorithm>
#include <atomic>
#include <thread>

#include "common.cuh"
#include "host_stage.h"

// minimal NCCL surface (types as in nccl.h 2.27/2.28; resolved at run time)
typedef struct { char internal[128]; } nimfm_ncclUniqueId;
typedef int (*fn_ncclGetUniqueId)(nimfm_ncclUniqueId *);
typedef int (*fn_ncclCommInitRank)(ncclComm **, int, nimfm_ncclUniqueId, int);
typedef int (*fn_ncclAllReduce)(const void *, void *, size_t, int, int, ncclComm *, cudaStream_t);
typedef int (*fn_ncclReduceScatter)(const void *, void *, size_t, int, int, ncclComm *, cudaStream_t);
typedef int (*fn_ncclAllGather)(const void *, void *, size_t, int, ncclComm *, cudaStream_t);
typedef int (*fn_ncclCommDestroy)(ncclComm *);
typedef const char *(*fn_ncclGetErrorString)(int);
static struct {
  void *h;
  fn_ncclGetUniqueId getUniqueId;
  fn_ncclCommInitRank commInitRank;
  fn_ncclAllReduce allReduce;
  fn_ncclReduceScatter reduceScatter;
  fn_ncclAllGather allGather;
  fn_ncclCommDestroy commDestroy;
  fn_ncclGetErrorString errStr;
} g_nccl;

static int load_nccl() {
  if (g_nccl.h) return 0;
  void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return -1;
  g_nccl.getUniqueId = (fn_ncclGetUniqueId)dlsym(h, "ncclGetUniqueId");
  g_nccl.commInitRank = (fn_ncclCommInitRank)dlsym(h, "ncclCommInitRank");
  g_nccl.allReduce = (fn_ncclAllReduce)dlsym(h, "ncclAllReduce");
  g_nccl.reduceScatter = (fn_ncclReduceScatter)dlsym(h, "ncclReduceScatter");
  g_nccl.allGather = (fn_ncclAllGather)dlsym(h, "ncclAllGather");
  g_nccl.commDestroy = (fn_ncclCommDestroy)dlsym(h, "ncclCommDestroy");
  g_nccl.errStr = (fn_ncclGetErrorString)dlsym(h, "ncclGetErrorString");
  if (!g_nccl.getUniqueId || !g_nccl.commInitRank || !g_nccl.allReduce || !g_nccl.commDestroy) return -1;
  g_nccl.h = h;
  return 0;
}

static thread_local std::string g_noctx_err;

int nimfm_fail(nimfm_ctx *ctx, int code, const char *fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  else g_noctx_err = buf;
  return code;
}

static int ctx_init_resources(nimfm_ctx *ctx) {
  CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  CK(cudaEventCreate(&ctx->ev0));
  CK(cudaEventCreate(&ctx->ev1));
  CK(cudaEventCreate(&ctx->tev0));
  CK(cudaEventCreate(&ctx->tev1));
  CK(cudaStreamCreateWithFlags(&ctx->copyStream, cudaStreamNonBlocking));
  for (int s = 0; s < 2; s++) {
    CK(cudaEventCreateWithFlags(&ctx->evCopied[s], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ctx->evComputed[s], cudaEventDisableTiming));
  }
  CK(cudaMalloc(&ctx->scalars, 64 * sizeof(double)));
  CK(cudaMemset(ctx->scalars, 0, 64 * sizeof(double)));
  CK(cudaMallocHost(&ctx->hostScalars, 64 * sizeof(double)));
  return NIMFM_OK;
}

extern "C" {

int32_t nimfm_version(void) { return 100; }

const char *nimfm_last_error(const nimfm_ctx *ctx) { return ctx ? ctx->err.c_str() : g_noctx_err.c_str(); }

int64_t nimfm_launch_count(const nimfm_ctx *ctx) { return ctx ? ctx->launches : 0; }
int32_t nimfm_mem_info(nimfm_ctx *ctx, int64_t *freeBytes, int64_t *totalBytes) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  size_t f = 0, t = 0;
  CK(cudaMemGetInfo(&f, &t));
  if (freeBytes) *freeBytes = (int64_t)f;
  if (totalBytes) *totalBytes = (int64_t)t;
  return NIMFM_OK;
}
int32_t nimfm_stream_stats(const nimfm_ctx *ctx, int64_t *h2dBytes, int64_t *d2hBytes, int32_t *hostThreads) {
  if (!ctx) return NIMFM_ERR_INVALID;
  if (h2dBytes) *h2dBytes = ctx->lastH2D;
  if (d2hBytes) *d2hBytes = ctx->lastD2H;
  if (hostThreads) *hostThreads = ctx->lastHostThreads;
  return NIMFM_OK;
}

int32_t nimfm_ctx_create(int32_t device, nimfm_ctx **out) {
  nimfm_ctx *ctx = nullptr;
  if (!out) return nimfm_fail(nullptr, NIMFM_ERR_INVALID, "out is NULL");
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return nimfm_fail(nullptr, NIMFM_ERR_CUDA,
                      "no CUDA device available (%s); libnimfm_cuda has no CPU fallback",
                      e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
  if (device < 0 || device >= count)
    return nimfm_fail(nullptr, NIMFM_ERR_INVALID, "device %d out of range [0,%d)", device, count);
  ctx = new nimfm_ctx();
  ctx->device = device;
  cudaDeviceProp prop;
  if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
    delete ctx;
    return nimfm_fail(nullptr, NIMFM_ERR_CUDA, "cannot select device %d", device);
  }
  if (prop.major < 10) {
    int maj = prop.major, mnr = prop.minor;
    delete ctx;
    return nimfm_fail(nullptr, NIMFM_ERR_UNSUPPORTED,
                      "device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, maj, mnr);
  }
  ctx->numSMs = prop.multiProcessorCount;
  ctx->smemOptin = (int)prop.sharedMemPerBlockOptin;
  ctx->smemPerSM = (int)prop.sharedMemPerMultiprocessor;
  const int rc = ctx_init_resources(ctx);
  if (rc != NIMFM_OK) {   // the half-built context is released; its message moves to the no-context slot
    const std::string msg = ctx->err;
    nimfm_ctx_destroy(ctx);
    return nimfm_fail(nullptr, rc, "%s", msg.c_str());
  }
  *out = ctx;
  return NIMFM_OK;
}

int32_t nimfm_ctx_destroy(nimfm_ctx *ctx) {
  if (!ctx) return NIMFM_OK;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  nimfm_peer_shutdown(ctx);
  if (ctx->comm && g_nccl.commDestroy) g_nccl.commDestroy(ctx->comm);
  cudaFree(ctx->partials);
  cudaFree(ctx->stash);
  nimfm_mb_index_free(ctx->mbIndex);
  cudaFree(ctx->scalars);
  cudaFree(ctx->idxScratch);
  cudaFree(ctx->idx32Scratch);
  cudaFreeHost(ctx->hostScalars);
  for (int s = 0; s < 2; s++) {
    cudaFree(ctx->stage[s].packed); cudaFree(ctx->stage[s].mask); cudaFree(ctx->stage[s].blk);
    cudaFree(ctx->stage[s].data); cudaFree(ctx->stage[s].y); cudaFree(ctx->stage[s].idx64);
    cudaFree(ctx->stage[s].indptr); cudaFree(ctx->stage[s].idx32);
    if (ctx->evCopied[s]) cudaEventDestroy(ctx->evCopied[s]);
    if (ctx->evComputed[s]) cudaEventDestroy(ctx->evComputed[s]);
  }
  for (int s = 0; s < nimfm_ctx::kPinPieces; s++) {
    if (ctx->pinPiece[s]) cudaFreeHost(ctx->pinPiece[s]);
    if (ctx->evPiece[s]) cudaEventDestroy(ctx->evPiece[s]);
  }
  for (int s = 0; s < 4; s++) {
    if (ctx->hostIdx[s]) cudaFreeHost(ctx->hostIdx[s]);
    if (ctx->hostPtr[s]) cudaFreeHost(ctx->hostPtr[s]);
    if (ctx->hostData[s]) cudaFreeHost(ctx->hostData[s]);
    if (ctx->hostPack[s]) cudaFreeHost(ctx->hostPack[s]);
    if (ctx->hostMask[s]) cudaFreeHost(ctx->hostMask[s]);
    if (ctx->hostBlk[s]) cudaFreeHost(ctx->hostBlk[s]);
    if (ctx->hostY[s]) cudaFreeHost(ctx->hostY[s]);
    if (ctx->evSlot[s]) cudaEventDestroy(ctx->evSlot[s]);
  }
  cudaFree(ctx->stageHotSlot);
  cudaFree(ctx->stageHotList);
  if (ctx->tev0) cudaEventDestroy(ctx->tev0);
  if (ctx->tev1) cudaEventDestroy(ctx->tev1);
  if (ctx->copyStream) cudaStreamDestroy(ctx->copyStream);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0);
  if (ctx->ev1) cudaEventDestroy(ctx->ev1);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return NIMFM_OK;
}

// Page-lock a caller-owned host array for the lifetime of the data set it belongs to (the Nim dataset object
// owns its seqs, so the lifetime is known there): host-fed calls then DMA straight out of it at link rate.
// Unregister before the array is freed or resized.
int32_t nimfm_host_register(nimfm_ctx *ctx, const void *ptr, int64_t bytes) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(ptr != nullptr && bytes > 0, "bad arguments");
  CK(cudaSetDevice(ctx->device));
  cudaError_t e = cudaHostRegister(const_cast<void *>(ptr), (size_t)bytes, cudaHostRegisterDefault);
  if (e == cudaErrorHostMemoryAlreadyRegistered) {
    cudaGetLastError();
    return NIMFM_OK;
  }
  if (e != cudaSuccess) return nimfm_fail(ctx, NIMFM_ERR_CUDA, "cudaHostRegister(%lld bytes): %s", (long long)bytes, cudaGetErrorString(e));
  return NIMFM_OK;
}

int32_t nimfm_host_unregister(nimfm_ctx *ctx, const void *ptr) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(ptr != nullptr, "ptr is NULL");
  CK(cudaSetDevice(ctx->device));
  cudaError_t e = cudaHostUnregister(const_cast<void *>(ptr));
  if (e == cudaErrorHostMemoryNotRegistered) {
    cudaGetLastError();
    return NIMFM_OK;
  }
  if (e != cudaSuccess) return nimfm_fail(ctx, NIMFM_ERR_CUDA, "cudaHostUnregister: %s", cudaGetErrorString(e));
  return NIMFM_OK;
}

int32_t nimfm_comm_unique_id(void *uid128) {
  if (!uid128) return nimfm_fail(nullptr, NIMFM_ERR_INVALID, "uid is NULL");
  if (load_nccl() != 0) return nimfm_fail(nullptr, NIMFM_ERR_NCCL, "cannot load libnccl.so.2: %s", dlerror());
  nimfm_ncclUniqueId id;
  int rc = g_nccl.getUniqueId(&id);
  if (rc != 0) return nimfm_fail(nullptr, NIMFM_ERR_NCCL, "ncclGetUniqueId: %s", g_nccl.errStr ? g_nccl.errStr(rc) : "?");
  memcpy(uid128, &id, 128);
  return NIMFM_OK;
}

int32_t nimfm_comm_init(nimfm_ctx *ctx, int32_t rank, int32_t nranks, const void *uid128) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, "bad rank %d / nranks %d", rank, nranks);
  ctx->rank = rank;
  ctx->nranks = nranks;
  if (nranks == 1) return NIMFM_OK;
  REQUIRE(uid128 != nullptr, "uid is NULL");
  if (load_nccl() != 0) return nimfm_fail(ctx, NIMFM_ERR_NCCL, "cannot load libnccl.so.2: %s", dlerror());
  CK(cudaSetDevice(ctx->device));
  nimfm_ncclUniqueId id;
  memcpy(&id, uid128, 128);
  int rc = g_nccl.commInitRank(&ctx->comm, nranks, id, rank);
  if (rc != 0) return nimfm_fail(ctx, NIMFM_ERR_NCCL, "ncclCommInitRank: %s", g_nccl.errStr ? g_nccl.errStr(rc) : "?");
  return nimfm_peer_init(ctx);   // NVLink peer-memory exchange (falls back to NCCL when the GPUs cannot map each other)
}

int32_t nimfm_comm_size(const nimfm_ctx *ctx) { return ctx ? ctx->nranks : 0; }

int32_t nimfm_comm_allgather_i64(nimfm_ctx *ctx, const int64_t *mine, int32_t count, int64_t *all) {
  if (!ctx) return NIMFM_ERR_INVALID;
  REQUIRE(mine && all && count >= 1 && count <= 4096, "bad arguments");
  CK(cudaSetDevice(ctx->device));
  return nimfm_allgather_host_i64(ctx, mine, count, all);
}

int32_t nimfm_timer_start(nimfm_ctx *ctx) {
  if (!ctx) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventRecord(ctx->tev0, ctx->stream));
  return NIMFM_OK;
}

int32_t nimfm_timer_stop(nimfm_ctx *ctx, float *ms) {
  if (!ctx || !ms) return NIMFM_ERR_INVALID;
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventRecord(ctx->tev1, ctx->stream));
  CK(cudaEventSynchronize(ctx->tev1));
  CK(cudaEventElapsedTime(ms, ctx->tev0, ctx->tev1));
  return NIMFM_OK;
}

}  // extern "C"

int nimfm_allreduce_sum(nimfm_ctx *ctx, double *buf, int64_t n) {
  if (ctx->nranks == 1) return NIMFM_OK;
  {   // buffers that live in a peer-mapped arena are reduced over NVLink peer memory (peer.cu), in a fixed rank order
    int done = 0;
    int rc = nimfm_peer_allreduce_sum(ctx, buf, n, &done);
    if (rc || done) return rc;
  }
  if (!ctx->comm) return nimfm_fail(ctx, NIMFM_ERR_NCCL, "communicator not initialised (nimfm_comm_init)");
  int rc = g_nccl.allReduce(buf, buf, (size_t)n, /*ncclDouble*/ 8, /*ncclSum*/ 0, ctx->comm, ctx->stream);
  if (rc != 0) return nimfm_fail(ctx, NIMFM_ERR_NCCL, "ncclAllReduce: %s", g_nccl.errStr ? g_nccl.errStr(rc) : "?");
  return NIMFM_OK;
}

// rank r receives the sum of elements [r*count, (r+1)*count) of every rank's buf, in place (at buf + r*count)
int nimfm_reduce_scatter_sum(nimfm_ctx *ctx, double *buf, int64_t count) {
  if (ctx->nranks == 1) return NIMFM_OK;
  if (!ctx->comm || !g_nccl.reduceScatter) return nimfm_fail(ctx, NIMFM_ERR_NCCL, "communicator not initialised (nimfm_comm_init)");
  int rc = g_nccl.reduceScatter(buf, buf + (int64_t)ctx->rank * count, (size_t)count, 8, 0, ctx->comm, ctx->stream);
  if (rc != 0) return nimfm_fail(ctx, NIMFM_ERR_NCCL, "ncclReduceScatter: %s", g_nccl.errStr ? g_nccl.errStr(rc) : "?");
  return NIMFM_OK;
}

// every rank's slice [r*count, (r+1)*count) of buf is distributed to all ranks, in place
int nimfm_allgather_inplace(nimfm_ctx *ctx, double *buf, int64_t count) {
  if (ctx->nranks == 1) return NIMFM_OK;
  if (!ctx->comm || !g_nccl.allGather) return nimfm_fail(ctx, NIMFM_ERR_NCCL, "communicator not initialised (nimfm_comm_init)");
  int rc = g_nccl.allGather(buf + (int64_t)ctx->rank * count, buf, (size_t)count, 8, ctx->comm, ctx->stream);
  if (rc != 0) return nimfm_fail(ctx, NIMFM_ERR_NCCL, "ncclAllGather: %s", g_nccl.errStr ? g_nccl.errStr(rc) : "?");
  return NIMFM_OK;
}

// `count` int64 values of every rank, rank-major, on every host (sizes the ranks must agree on before a
// sharded epoch: shard lengths, minibatch shares).  One rank: a copy.
int nimfm_allgather_host_i64(nimfm_ctx *ctx, const int64_t *mine, int count, int64_t *all) {
  if (ctx->nranks == 1) {
    memcpy(all, mine, (size_t)count * 8);
    return NIMFM_OK;
  }
  if (!ctx->comm || !g_nccl.allGather) return nimfm_fail(ctx, NIMFM_ERR_NCCL, "communicator not initialised (nimfm_comm_init)");
  int rc = nimfm_ensure_idx(ctx, (size_t)count * (ctx->nranks + 1));
  if (rc) return rc;
  int64_t *dAll = ctx->idxScratch, *dMine = ctx->idxScratch + (size_t)count * ctx->nranks;
  CK(cudaMemcpyAsync(dMine, mine, (size_t)count * 8, cudaMemcpyHostToDevice, ctx->stream));
  rc = g_nccl.allGather(dMine, dAll, (size_t)count, /*ncclInt64*/ 4, ctx->comm, ctx->stream);
  if (rc != 0) return nimfm_fail(ctx, NIMFM_ERR_NCCL, "ncclAllGather: %s", g_nccl.errStr ? g_nccl.errStr(rc) : "?");
  CK(cudaMemcpyAsync(all, dAll, (size_t)count * ctx->nranks * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return NIMFM_OK;
}

int nimfm_mb_schedule(nimfm_ctx *ctx, int64_t nRows, int64_t mb, int64_t it, MbSchedule *out) {
  const int R = ctx->nranks;
  out->rank = ctx->rank;
  out->nRows.assign((size_t)R, nRows);
  out->mb.assign((size_t)R, mb);
  if (R > 1) {
    const int64_t mine[3] = {nRows, mb, it};
    std::vector<int64_t> all((size_t)3 * R);
    int rc = nimfm_allgather_host_i64(ctx, mine, 3, all.data());
    if (rc) return rc;
    for (int r = 0; r < R; r++) {
      out->nRows[(size_t)r] = all[(size_t)3 * r];
      out->mb[(size_t)r] = all[(size_t)3 * r + 1];
      if (all[(size_t)3 * r + 2] != it)
        return nimfm_fail(ctx, NIMFM_ERR_STATE, "rank %d is at iteration %lld, rank %d at %lld: the replicas have diverged",
                          r, (long long)all[(size_t)3 * r + 2], ctx->rank, (long long)it);
      if (out->mb[(size_t)r] < 1) return nimfm_fail(ctx, NIMFM_ERR_INVALID, "rank %d has miniBatchSize < 1", r);
    }
  }
  out->T = 0;
  for (int r = 0; r < R; r++)
    out->T = std::max(out->T, (out->nRows[(size_t)r] + out->mb[(size_t)r] - 1) / out->mb[(size_t)r]);
  return NIMFM_OK;
}

void nimfm_trace_begin(nimfm_ctx *ctx, const char *tag) {
  if (ctx->traceOn < 0) { const char *e = getenv("NIMFM_TRACE"); ctx->traceOn = e && e[0] == '1'; }
  if (!ctx->traceOn) return;
  nimfm_ctx::TraceSpan sp{tag, nullptr, nullptr, true};
  cudaEventCreate(&sp.e0);
  cudaEventCreate(&sp.e1);
  cudaEventRecord(sp.e0, ctx->stream);
  ctx->trace.push_back(sp);
}
void nimfm_trace_end(nimfm_ctx *ctx) {
  if (ctx->traceOn != 1) return;
  for (auto sp = ctx->trace.rbegin(); sp != ctx->trace.rend(); ++sp)
    if (sp->open) {
      cudaEventRecord(sp->e1, ctx->stream);
      sp->open = false;
      return;
    }
}
void nimfm_trace_report(nimfm_ctx *ctx, const char *what) {
  if (ctx->traceOn != 1 || ctx->trace.empty()) return;
  cudaStreamSynchronize(ctx->stream);
  struct Acc { const char *tag; double ms; int n; };
  std::vector<Acc> acc;
  for (auto &sp : ctx->trace) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, sp.e0, sp.e1);
    cudaEventDestroy(sp.e0);
    cudaEventDestroy(sp.e1);
    bool found = false;
    for (auto &a : acc) if (!strcmp(a.tag, sp.tag)) { a.ms += ms; a.n++; found = true; }
    if (!found) acc.push_back({sp.tag, ms, 1});
  }
  ctx->trace.clear();
  std::string line = std::string("[nimfm trace] rank ") + std::to_string(ctx->rank) + " " + what + ":";
  for (auto &a : acc) {
    char buf[128];
    snprintf(buf, sizeof(buf), "  %s %.1f us x %d", a.tag, a.ms * 1e3 / a.n, a.n);
    line += buf;
  }
  fprintf(stderr, "%s\n", line.c_str());
}

int nimfm_ensure_partials(nimfm_ctx *ctx, size_t nDoubles) {
  if (ctx->partialsCap >= nDoubles) return NIMFM_OK;
  if (ctx->partials) {
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaFree(ctx->partials));
    ctx->partials = nullptr;
    ctx->partialsCap = 0;
  }
  size_t cap = nDoubles < 65536 ? 65536 : nDoubles;
  CK(cudaMalloc(&ctx->partials, cap * sizeof(double)));
  ctx->partialsCap = cap;
  return NIMFM_OK;
}

int nimfm_ensure_idx(nimfm_ctx *ctx, size_t n) {
  if (ctx->idxCap >= n) return NIMFM_OK;
  CK(cudaStreamSynchronize(ctx->stream));
  if (ctx->idxScratch) CK(cudaFree(ctx->idxScratch));
  if (ctx->idx32Scratch) CK(cudaFree(ctx->idx32Scratch));
  ctx->idxScratch = nullptr;
  ctx->idx32Scratch = nullptr;
  ctx->idxCap = 0;
  size_t cap = n < 4096 ? 4096 : n;
  CK(cudaMalloc(&ctx->idxScratch, cap * sizeof(int64_t)));
  CK(cudaMalloc(&ctx->idx32Scratch, cap * sizeof(int32_t)));
  ctx->idxCap = cap;
  return NIMFM_OK;
}

__global__ void narrow_ids_kernel(const int64_t *in, int32_t *out, int64_t count, int64_t n, int *bad) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t v = in[i];
    if (v < 0 || v >= n) { *bad = 1; v = 0; }
    out[i] = (int32_t)v;
  }
}

int nimfm_stage_row_ids(nimfm_ctx *ctx, const int64_t *ids, int64_t count, int64_t n) {
  int rc = nimfm_ensure_idx(ctx, (size_t)count + 2);
  if (rc) return rc;
  CK(cudaMemcpyAsync(ctx->idxScratch, ids, (size_t)count * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
  int *bad = reinterpret_cast<int *>(ctx->scalars + 60);
  CK(cudaMemsetAsync(bad, 0, sizeof(int), ctx->stream));
  int grid = (int)((count + 255) / 256);
  if (grid > 4096) grid = 4096;
  if (grid < 1) grid = 1;
  narrow_ids_kernel<<<grid, 256, 0, ctx->stream>>>(ctx->idxScratch, ctx->idx32Scratch, count, n, bad);
  LAUNCHED(ctx);
  int hbad = 0;
  CK(cudaMemcpyAsync(&hbad, bad, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  if (hbad) return nimfm_fail(ctx, NIMFM_ERR_INVALID, "row index out of range [0,%lld)", (long long)n);
  return NIMFM_OK;
}

// Pageable host memory (a caller's numpy / Nim seq arrays, an mmap'ed file) -> device.  cudaMemcpy from
// pageable memory runs at ~4 GB/s here (the driver stages it through one pinned bounce buffer on one
// thread); a team of threads copying 8 MB pieces into the context's pinned pieces, each thread issuing the
// async copy of the piece it just filled, keeps the link busy instead.  With narrowD > 0 the source is
// int64 ids and the pieces are filled with their int32 narrowing (range-checked against [0, narrowD):
// *bad is set, the caller reports).  The context's stream waits for the last piece.
int nimfm_staged_h2d(nimfm_ctx *ctx, void *dDst, const void *srcv, size_t bytes, int64_t narrowD, int *bad) {
  if (bad) *bad = 0;
  if (bytes == 0) return NIMFM_OK;
  const char *src = static_cast<const char *>(srcv);
  const bool narrowing = narrowD > 0;
  const size_t piece = nimfm_ctx::kPinPieceBytes;            // bytes of DESTINATION per piece
  const size_t dstBytes = narrowing ? bytes / 2 : bytes;
  const int64_t nPieces = (int64_t)((dstBytes + piece - 1) / piece);
  const int hw = (int)std::thread::hardware_concurrency();
  int T = (int)std::min<int64_t>(std::min(8, std::max(1, hw / std::max(1, ctx->nranks))), nPieces);
  if (const char *e = getenv("NIMFM_HOST_THREADS")) T = std::max(1, std::min(atoi(e), 8));
  for (int i = 0; i < nimfm_ctx::kPinPieces; i++) {
    if (!ctx->pinPiece[i]) CK(cudaHostAlloc(&ctx->pinPiece[i], piece, cudaHostAllocDefault));
    if (!ctx->evPiece[i]) CK(cudaEventCreateWithFlags(&ctx->evPiece[i], cudaEventDisableTiming));
  }
  std::atomic<int64_t> next(0);
  std::atomic<int> err((int)cudaSuccess), anyBad(0);
  auto work = [&](int t) {
    if (cudaSetDevice(ctx->device) != cudaSuccess) { err = (int)cudaErrorInvalidDevice; return; }
    int use = 0;   // thread t owns pieces 2t and 2t+1 of the pinned set
    for (;;) {
      const int64_t i = next.fetch_add(1);
      if (i >= nPieces || err.load() != (int)cudaSuccess) return;
      const int slot = 2 * t + (use++ & 1);
      const size_t off = (size_t)i * piece, len = std::min(piece, dstBytes - off);
      cudaError_t e = cudaEventSynchronize(ctx->evPiece[slot]);   // the slot's previous copy has left the host
      if (narrowing) {
        if (nimfm_host_narrow(reinterpret_cast<const int64_t *>(src) + off / 4,
                              reinterpret_cast<int32_t *>(ctx->pinPiece[slot]), (int64_t)(len / 4), narrowD))
          anyBad = 1;
      } else {
        memcpy(ctx->pinPiece[slot], src + off, len);
      }
      if (e == cudaSuccess)
        e = cudaMemcpyAsync(static_cast<char *>(dDst) + off, ctx->pinPiece[slot], len, cudaMemcpyHostToDevice, ctx->copyStream);
      if (e == cudaSuccess) e = cudaEventRecord(ctx->evPiece[slot], ctx->copyStream);
      if (e != cudaSuccess) { err = (int)e; return; }
    }
  };
  if (T < 2 || nPieces < 2) {
    work(0);
  } else {
    std::vector<std::thread> team;
    for (int t = 0; t < T; t++) team.emplace_back(work, t);
    for (auto &th : team) th.join();
  }
  if (err.load() != (int)cudaSuccess)
    return nimfm_fail(ctx, NIMFM_ERR_CUDA, "staged_h2d: %s", cudaGetErrorString((cudaError_t)err.load()));
  if (bad) *bad = anyBad.load();
  CK(cudaEventRecord(ctx->evCopied[0], ctx->copyStream));
  CK(cudaStreamWaitEvent(ctx->stream, ctx->evCopied[0], 0));
  return NIMFM_OK;
}

// Device -> pageable host memory, the same way round: every thread queues the async copy of a piece into
// one of its pinned slots, waits for it, and copies it out while the other threads' pieces are on the link.
// Everything queued on the context's stream before the call is waited for; the call returns with the data
// in place.
int nimfm_staged_d2h(nimfm_ctx *ctx, void *hostDst, const void *dSrc, size_t bytes) {
  if (bytes == 0) return NIMFM_OK;
  const size_t piece = nimfm_ctx::kPinPieceBytes;
  const int64_t nPieces = (int64_t)((bytes + piece - 1) / piece);
  const int hw = (int)std::thread::hardware_concurrency();
  int T = (int)std::min<int64_t>(std::min(8, std::max(1, hw / std::max(1, ctx->nranks))), nPieces);
  if (const char *e = getenv("NIMFM_HOST_THREADS")) T = std::max(1, std::min(atoi(e), 8));
  for (int i = 0; i < nimfm_ctx::kPinPieces; i++) {
    if (!ctx->pinPiece[i]) CK(cudaHostAlloc(&ctx->pinPiece[i], piece, cudaHostAllocDefault));
    if (!ctx->evPiece[i]) CK(cudaEventCreateWithFlags(&ctx->evPiece[i], cudaEventDisableTiming));
  }
  CK(cudaEventRecord(ctx->evComputed[0], ctx->stream));
  CK(cudaStreamWaitEvent(ctx->copyStream, ctx->evComputed[0], 0));
  std::atomic<int64_t> next(0);
  std::atomic<int> err((int)cudaSuccess);
  auto work = [&](int t) {
    if (cudaSetDevice(ctx->device) != cudaSuccess) { err = (int)cudaErrorInvalidDevice; return; }
    const int slot = 2 * t;
    for (;;) {
      const int64_t i = next.fetch_add(1);
      if (i >= nPieces || err.load() != (int)cudaSuccess) return;
      const size_t off = (size_t)i * piece, len = std::min(piece, bytes - off);
      cudaError_t e = cudaEventSynchronize(ctx->evPiece[slot]);   // an earlier H2D out of this slot has left
      if (e == cudaSuccess)
        e = cudaMemcpyAsync(ctx->pinPiece[slot], static_cast<const char *>(dSrc) + off, len, cudaMemcpyDeviceToHost, ctx->copyStream);
      if (e == cudaSuccess) e = cudaEventRecord(ctx->evPiece[slot], ctx->copyStream);
      if (e == cudaSuccess) e = cudaEventSynchronize(ctx->evPiece[slot]);
      if (e != cudaSuccess) { err = (int)e; return; }
      memcpy(static_cast<char *>(hostDst) + off, ctx->pinPiece[slot], len);
    }
  };
  if (T < 2 || nPieces < 2) {
    work(0);
  } else {
    std::vector<std::thread> team;
    for (int t = 0; t < T; t++) team.emplace_back(work, t);
    for (auto &th : team) th.join();
  }
  if (err.load() != (int)cudaSuccess)
    return nimfm_fail(ctx, NIMFM_ERR_CUDA, "staged_d2h: %s", cudaGetErrorString((cudaError_t)err.load()));
  return NIMFM_OK;
}
