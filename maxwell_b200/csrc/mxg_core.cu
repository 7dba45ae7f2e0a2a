// libmxgpu: context, maps, multivector lifetime and transfers.
#include <cstdlib>
#include <cstring>

#include "mxg_internal.h"

namespace mxg {
static thread_local char g_err[1024] = "";
void setError(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int ensureScratch(mxg_ctx* ctx, size_t bytes) {
  if (ctx->scratchBytes >= bytes) return MXG_OK;
  if (ctx->dScratch) MXG_CUDA(cudaFree(ctx->dScratch));
  ctx->dScratch = nullptr;
  ctx->scratchBytes = 0;
  size_t want = bytes < (1u << 20) ? (1u << 20) : bytes;
  MXG_CUDA(cudaMalloc(&ctx->dScratch, want));
  ctx->scratchBytes = want;
  return MXG_OK;
}
int ensurePinned(mxg_ctx* ctx, size_t bytes) {
  if (ctx->pinnedBytes >= bytes) return MXG_OK;
  if (ctx->hPinned) MXG_CUDA(cudaFreeHost(ctx->hPinned));
  ctx->hPinned = nullptr;
  ctx->pinnedBytes = 0;
  size_t want = bytes < (1u << 20) ? (1u << 20) : bytes;
  MXG_CUDA(cudaMallocHost(&ctx->hPinned, want));
  ctx->pinnedBytes = want;
  return MXG_OK;
}
int allReduceScratch(mxg_ctx* ctx, size_t count) {
  if (ctx->nranks <= 1) return MXG_OK;
  MXG_REQUIRE(ctx->comm != nullptr, "communicator not initialised");
  MXG_NCCL(ncclAllReduce(ctx->dScratch, ctx->dScratch, count, ncclDouble, ncclSum, ctx->comm, ctx->stream));
  return MXG_OK;
}
int checkHaloFault(const mxg_ctx* ctx, const char* where) {
  MXG_REQUIRE(!ctx->hErr || *ctx->hErr == 0, "%s: a halo exchange timed out waiting for a neighbour rank (dead or dead-locked rank)", where);
  return MXG_OK;
}
int mapGlobalCount(mxg_map* map, int64_t* out) {
  if (map->nMapGlobal < 0) {
    mxg_ctx* ctx = map->ctx;
    int64_t cnt = map->nLocal;
    if (ctx->nranks > 1) {
      MXG_REQUIRE(ctx->comm != nullptr, "communicator not initialised");
      int64_t* d = nullptr;
      MXG_CUDA(cudaMalloc(&d, sizeof(int64_t)));
      MXG_CUDA(cudaMemcpyAsync(d, &cnt, sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
      MXG_NCCL(ncclAllReduce(d, d, 1, ncclInt64, ncclSum, ctx->comm, ctx->stream));
      MXG_CUDA(cudaMemcpyAsync(&cnt, d, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
      MXG_CUDA(cudaStreamSynchronize(ctx->stream));
      MXG_CUDA(cudaFree(d));
    }
    map->nMapGlobal = cnt;
  }
  *out = map->nMapGlobal;
  return MXG_OK;
}
}  // namespace mxg

MvStorage::~MvStorage() {
  if (base) {
    cudaSetDevice(ctx->device);
    cudaFree(base);
  }
}

using namespace mxg;

namespace {
static int ctxInit(mxg_ctx* ctx, int device) {
  ctx->device = device;
  ctx->graphsOff = std::getenv("MXG_NO_GRAPH") != nullptr;   // eager enqueues instead of graph replay
  MXG_CUDA(cudaDeviceGetAttribute(&ctx->numSMs, cudaDevAttrMultiProcessorCount, device));
  MXG_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  {
    // halo exchange + boundary rows get scheduling priority over the bulk interior rows
    int lo = 0, hi = 0;
    MXG_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    MXG_CUDA(cudaStreamCreateWithPriority(&ctx->commStream, cudaStreamNonBlocking, hi));
  }
  MXG_CUDA(cudaEventCreateWithFlags(&ctx->evA, cudaEventDisableTiming));
  MXG_CUDA(cudaEventCreateWithFlags(&ctx->evB, cudaEventDisableTiming));
  MXG_CUDA(cudaHostAlloc(&ctx->hErr, sizeof(int), cudaHostAllocMapped));
  *ctx->hErr = 0;
  MXG_CUDA(cudaHostGetDevicePointer(&ctx->dErr, ctx->hErr, 0));
  {
    double seconds = 120.0;
    if (const char* e = std::getenv("MXG_HALO_TIMEOUT_S")) seconds = std::atof(e);
    int khz = 0;
    MXG_CUDA(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device));
    ctx->haloTimeoutTicks = seconds > 0 ? (long long)(seconds * 1e3 * double(khz)) : 0;
  }
  MXG_CUDA(cudaMalloc(&ctx->dDense, 64 * 1024));
  int rc = ensureScratch(ctx, 1u << 20);
  if (rc) return rc;
  return ensurePinned(ctx, 1u << 20);
}

}  // namespace

extern "C" {

const char* mxg_last_error(void) { return g_err; }
int mxg_version(void) { return 100; }

int mxg_ctx_create(int device, mxg_ctx** out) {
  MXG_REQUIRE(out != nullptr, "mxg_ctx_create: out is NULL");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    setError("mxg_ctx_create: no CUDA device available (%s); libmxgpu has no CPU fallback",
             e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    return MXG_ERR_CUDA;
  }
  MXG_REQUIRE(device >= 0 && device < ndev, "mxg_ctx_create: device %d out of range (0..%d)", device, ndev - 1);
  MXG_CUDA(cudaSetDevice(device));
  mxg_ctx* ctx = new mxg_ctx;
  const int rc = ctxInit(ctx, device);
  if (rc) {   // one cleanup path: whatever was created so far is released
    mxg_ctx_destroy(ctx);
    return rc;
  }
  *out = ctx;
  return MXG_OK;
}

int mxg_ctx_destroy(mxg_ctx* ctx) {
  if (!ctx) return MXG_OK;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->commStream) cudaStreamSynchronize(ctx->commStream);
  if (ctx->comm) ncclCommDestroy(ctx->comm);
  if (ctx->dScratch) cudaFree(ctx->dScratch);
  if (ctx->dDense) cudaFree(ctx->dDense);
  if (ctx->hPinned) cudaFreeHost(ctx->hPinned);
  if (ctx->hErr) cudaFreeHost(ctx->hErr);
  if (ctx->evA) cudaEventDestroy(ctx->evA);
  if (ctx->evB) cudaEventDestroy(ctx->evB);
  for (auto& e : ctx->timer)
    if (e) cudaEventDestroy(e);
  for (auto& e : ctx->prof)
    if (e) cudaEventDestroy(e);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->commStream) cudaStreamDestroy(ctx->commStream);
  delete ctx;
  return MXG_OK;
}

int mxg_ctx_sync(mxg_ctx* ctx) {
  MXG_REQUIRE(ctx != nullptr, "mxg_ctx_sync: ctx is NULL");
  const cudaError_t e1 = cudaStreamSynchronize(ctx->commStream), e2 = cudaStreamSynchronize(ctx->stream);
  int rc = checkHaloFault(ctx, "mxg_ctx_sync");
  if (rc) return rc;
  MXG_CUDA(e1);
  MXG_CUDA(e2);
  return MXG_OK;
}
uint64_t mxg_ctx_random_epoch(mxg_ctx* ctx) { return ctx ? ctx->randomEpoch++ : 0; }
int mxg_ctx_rank(const mxg_ctx* ctx) { return ctx ? ctx->rank : 0; }
int mxg_ctx_num_ranks(const mxg_ctx* ctx) { return ctx ? ctx->nranks : 1; }
void* mxg_ctx_stream(mxg_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
int64_t mxg_ctx_launch_count(const mxg_ctx* ctx) { return ctx ? ctx->launches : 0; }

int mxg_ctx_event_record(mxg_ctx* ctx, int slot) {
  MXG_REQUIRE(ctx && slot >= 0 && slot < 16, "mxg_ctx_event_record: bad slot %d", slot);
  MXG_CUDA(cudaSetDevice(ctx->device));
  if (!ctx->timer[slot]) MXG_CUDA(cudaEventCreate(&ctx->timer[slot]));
  MXG_CUDA(cudaEventRecord(ctx->timer[slot], ctx->stream));
  return MXG_OK;
}
int mxg_ctx_event_elapsed_ms(mxg_ctx* ctx, int a, int b, double* ms) {
  MXG_REQUIRE(ctx && ms && a >= 0 && a < 16 && b >= 0 && b < 16, "mxg_ctx_event_elapsed_ms: bad argument");
  MXG_REQUIRE(ctx->timer[a] && ctx->timer[b], "mxg_ctx_event_elapsed_ms: slot not recorded");
  MXG_CUDA(cudaEventSynchronize(ctx->timer[b]));
  float f = 0;
  MXG_CUDA(cudaEventElapsedTime(&f, ctx->timer[a], ctx->timer[b]));
  *ms = f;
  return MXG_OK;
}
void* mxg_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) {
    setError("mxg_host_alloc: cudaMallocHost(%zu) failed", bytes);
    return nullptr;
  }
  return p;
}
void mxg_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

int mxg_comm_unique_id(void* out) {
  MXG_REQUIRE(out != nullptr, "mxg_comm_unique_id: out is NULL");
  static_assert(sizeof(ncclUniqueId) <= MXG_UNIQUE_ID_BYTES, "unique id does not fit");
  ncclUniqueId id;
  MXG_NCCL(ncclGetUniqueId(&id));
  std::memset(out, 0, MXG_UNIQUE_ID_BYTES);
  std::memcpy(out, &id, sizeof(id));
  return MXG_OK;
}

int mxg_ctx_comm_init(mxg_ctx* ctx, int rank, int nranks, const void* unique_id) {
  MXG_REQUIRE(ctx != nullptr, "mxg_ctx_comm_init: ctx is NULL");
  MXG_REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, "mxg_ctx_comm_init: bad rank %d of %d", rank, nranks);
  MXG_REQUIRE(ctx->comm == nullptr, "mxg_ctx_comm_init: communicator already initialised");
  ctx->rank = rank;
  ctx->nranks = nranks;
  if (nranks == 1) return MXG_OK;
  MXG_REQUIRE(unique_id != nullptr, "mxg_ctx_comm_init: unique_id is NULL");
  MXG_CUDA(cudaSetDevice(ctx->device));
  ncclUniqueId id;
  std::memcpy(&id, unique_id, sizeof(id));
  MXG_NCCL(ncclCommInitRank(&ctx->comm, nranks, id, rank));
  return MXG_OK;
}

// ---- maps ------------------------------------------------------------------------------
int mxg_map_create(mxg_ctx* ctx, int64_t n_global, const int64_t* my_gids, int64_t n_local, mxg_map** out) {
  MXG_REQUIRE(ctx && out, "mxg_map_create: NULL argument");
  MXG_REQUIRE(n_local >= 0 && n_global >= n_local, "mxg_map_create: bad sizes (local %lld, global %lld)",
              (long long)n_local, (long long)n_global);
  MXG_REQUIRE(n_local < (int64_t(1) << 31), "mxg_map_create: local size must fit in 31 bits");
  MXG_REQUIRE(n_local == 0 || my_gids != nullptr, "mxg_map_create: my_gids is NULL");
  for (int64_t i = 1; i < n_local; ++i)
    MXG_REQUIRE(my_gids[i] > my_gids[i - 1], "mxg_map_create: GIDs must be strictly ascending (position %lld)", (long long)i);
  MXG_CUDA(cudaSetDevice(ctx->device));
  mxg_map* m = new mxg_map;
  m->ctx = ctx;
  m->nGlobal = n_global;
  m->nLocal = n_local;
  m->gids.assign(my_gids, my_gids + n_local);
  if (n_local > 0) {
    MXG_CUDA(cudaMalloc(&m->dGids, n_local * sizeof(int64_t)));
    MXG_CUDA(cudaMemcpyAsync(m->dGids, my_gids, n_local * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    MXG_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  *out = m;
  return MXG_OK;
}

static void mapRelease(mxg_map* m) {
  if (--m->refs == 0) {
    cudaSetDevice(m->ctx->device);
    if (m->dGids) cudaFree(m->dGids);
    delete m;
  }
}
int mxg_map_destroy(mxg_map* map) {
  if (map) mapRelease(map);
  return MXG_OK;
}
int64_t mxg_map_local_size(const mxg_map* map) { return map ? map->nLocal : -1; }
int64_t mxg_map_global_size(const mxg_map* map) { return map ? map->nGlobal : -1; }

// ---- multivector lifetime --------------------------------------------------------------
static int allocMv(mxg_map* map, int ncols, bool isComplex, bool zero, mxg_mv** out) {
  MXG_REQUIRE(map && out, "multivector: NULL argument");
  MXG_REQUIRE(ncols >= 1 && ncols <= MXG_MAX_COLS, "multivector: ncols %d outside 1..%d", ncols, MXG_MAX_COLS);
  mxg_ctx* ctx = map->ctx;
  MXG_CUDA(cudaSetDevice(ctx->device));
  const size_t esz = isComplex ? 16 : 8;
  // columns start on 256-byte boundaries (the bulk copies of the windowed SpMM need 16-byte aligned sources; kernels
  // take column pointers, so the stride is invisible outside this file)
  const size_t colBytes = (size_t(map->nLocal) * esz + 255) / 256 * 256;
  const size_t bytes = colBytes * ncols;
  auto st = std::make_shared<MvStorage>();
  st->ctx = ctx;
  st->bytes = bytes;
  if (bytes) {
    MXG_CUDA(cudaMalloc(&st->base, bytes));
    if (zero) MXG_CUDA(cudaMemsetAsync(st->base, 0, bytes, ctx->stream));
  }
  mxg_mv* mv = new mxg_mv;
  mv->map = map;
  map->refs++;
  mv->isComplex = isComplex;
  mv->ncols = ncols;
  mv->ld = map->nLocal;
  mv->storage = st;
  mv->col.resize(ncols);
  mv->baseCol.resize(ncols);
  for (int j = 0; j < ncols; ++j) {
    mv->col[j] = static_cast<char*>(st->base) + size_t(j) * colBytes;
    mv->baseCol[j] = j;
  }
  *out = mv;
  return MXG_OK;
}

int mxg_mv_create(mxg_map* map, int ncols, int is_complex, mxg_mv** out) {
  return allocMv(map, ncols, is_complex != 0, true, out);
}

int mxg_mv_view(mxg_mv* parent, const int* cols, int ncols, mxg_mv** out) {
  MXG_REQUIRE(parent && out, "mxg_mv_view: NULL argument");
  MXG_REQUIRE(ncols >= 1 && ncols <= MXG_MAX_COLS && cols, "mxg_mv_view: bad column list");
  for (int j = 0; j < ncols; ++j)
    MXG_REQUIRE(cols[j] >= 0 && cols[j] < parent->ncols, "mxg_mv_view: column %d out of range", cols[j]);
  mxg_mv* mv = new mxg_mv;
  mv->map = parent->map;
  mv->map->refs++;
  mv->isComplex = parent->isComplex;
  mv->ncols = ncols;
  mv->ld = parent->ld;
  mv->storage = parent->storage;
  mv->col.resize(ncols);
  mv->baseCol.resize(ncols);
  for (int j = 0; j < ncols; ++j) {
    mv->col[j] = parent->col[cols[j]];
    mv->baseCol[j] = parent->baseCol[cols[j]];
  }
  *out = mv;
  return MXG_OK;
}

int mxg_mv_clone_copy(const mxg_mv* src, const int* cols, int ncols, mxg_mv** out) {
  MXG_REQUIRE(src && out, "mxg_mv_clone_copy: NULL argument");
  if (!cols) ncols = src->ncols;
  MXG_REQUIRE(ncols >= 1 && ncols <= MXG_MAX_COLS, "mxg_mv_clone_copy: bad column count %d", ncols);
  mxg_mv* mv = nullptr;
  int rc = allocMv(src->map, ncols, src->isComplex, false, &mv);
  if (rc) return rc;
  mxg_ctx* ctx = src->map->ctx;
  const size_t colBytes = size_t(src->ld) * (src->isComplex ? 16 : 8);
  for (int j = 0; j < ncols; ++j) {
    const int s = cols ? cols[j] : j;
    if (s < 0 || s >= src->ncols) {
      mxg_mv_destroy(mv);
      setError("mxg_mv_clone_copy: column %d out of range", s);
      return MXG_ERR_ARG;
    }
    if (colBytes) MXG_CUDA(cudaMemcpyAsync(mv->col[j], src->col[s], colBytes, cudaMemcpyDeviceToDevice, ctx->stream));
  }
  *out = mv;
  return MXG_OK;
}

int mxg_mv_destroy(mxg_mv* mv) {
  if (!mv) return MXG_OK;
  mxg_map* m = mv->map;
  // storage may be freed here: make sure no queued kernel still uses it
  if (mv->storage.use_count() == 1) cudaStreamSynchronize(m->ctx->stream);
  delete mv;
  mapRelease(m);
  return MXG_OK;
}

int mxg_mv_num_cols(const mxg_mv* mv) { return mv ? mv->ncols : -1; }
int64_t mxg_mv_local_length(const mxg_mv* mv) { return mv ? mv->ld : -1; }
int64_t mxg_mv_global_length(const mxg_mv* mv) { return mv ? mv->map->nGlobal : -1; }
int mxg_mv_is_complex(const mxg_mv* mv) { return mv ? int(mv->isComplex) : -1; }
mxg_map* mxg_mv_get_map(const mxg_mv* mv) { return mv ? mv->map : nullptr; }
mxg_map* mxg_crs_row_map(const mxg_crs* A) { return A ? A->rowMap : nullptr; }
mxg_map* mxg_crs_domain_map(const mxg_crs* A) { return A ? A->domMap : nullptr; }
void* mxg_mv_col_ptr(mxg_mv* mv, int j) { return (mv && j >= 0 && j < mv->ncols) ? mv->col[j] : nullptr; }

int mxg_mv_upload(mxg_mv* mv, const double* host, int64_t ld) {
  MXG_REQUIRE(mv && host, "mxg_mv_upload: NULL argument");
  MXG_REQUIRE(ld >= mv->ld, "mxg_mv_upload: ld %lld smaller than local length %lld", (long long)ld, (long long)mv->ld);
  mxg_ctx* ctx = mv->map->ctx;
  const size_t esz = mv->isComplex ? 16 : 8;
  for (int j = 0; j < mv->ncols; ++j)
    if (mv->ld)
      MXG_CUDA(cudaMemcpyAsync(mv->col[j], reinterpret_cast<const char*>(host) + size_t(j) * ld * esz, mv->ld * esz,
                               cudaMemcpyHostToDevice, ctx->stream));
  MXG_CUDA(cudaStreamSynchronize(ctx->stream));
  return MXG_OK;
}

int mxg_mv_download(const mxg_mv* mv, double* host, int64_t ld) {
  MXG_REQUIRE(mv && host, "mxg_mv_download: NULL argument");
  MXG_REQUIRE(ld >= mv->ld, "mxg_mv_download: ld %lld smaller than local length %lld", (long long)ld, (long long)mv->ld);
  mxg_ctx* ctx = mv->map->ctx;
  const size_t esz = mv->isComplex ? 16 : 8;
  for (int j = 0; j < mv->ncols; ++j)
    if (mv->ld)
      MXG_CUDA(cudaMemcpyAsync(reinterpret_cast<char*>(host) + size_t(j) * ld * esz, mv->col[j], mv->ld * esz,
                               cudaMemcpyDeviceToHost, ctx->stream));
  {
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    int rc = checkHaloFault(ctx, "mxg_mv_download");
    if (rc) return rc;
    MXG_CUDA(e);
  }
  return MXG_OK;
}

}  // extern "C"
