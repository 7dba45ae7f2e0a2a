// Internal declarations shared by the libmxgpu translation units. sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <nccl.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <memory>
#include <string>
#include <vector>

#include "mxgpu.h"

namespace mxg {

void setError(const char* fmt, ...);

#define MXG_CUDA(expr)                                                                       \
  do {                                                                                       \
    cudaError_t e_ = (expr);                                                                 \
    if (e_ != cudaSuccess) {                                                                 \
      mxg::setError("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e_)); \
      return MXG_ERR_CUDA;                                                                   \
    }                                                                                        \
  } while (0)

#define MXG_NCCL(expr)                                                                       \
  do {                                                                                       \
    ncclResult_t r_ = (expr);                                                                \
    if (r_ != ncclSuccess) {                                                                 \
      mxg::setError("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, ncclGetErrorString(r_)); \
      return MXG_ERR_NCCL;                                                                   \
    }                                                                                        \
  } while (0)

#define MXG_REQUIRE(cond, ...)      \
  do {                              \
    if (!(cond)) {                  \
      mxg::setError(__VA_ARGS__);   \
      return MXG_ERR_ARG;           \
    }                               \
  } while (0)

// complex128 on the device: plain (re, im) pair, bit-compatible with std::complex<double>
struct __align__(16) zd {
  double x, y;
};
#ifdef __CUDACC__
__device__ __forceinline__ double ldgT(const double* p) { return __ldg(p); }
__device__ __forceinline__ zd ldgT(const zd* p) {
  const double2 v = __ldg(reinterpret_cast<const double2*>(p));
  return {v.x, v.y};
}
#endif
__host__ __device__ inline zd operator+(zd a, zd b) { return {a.x + b.x, a.y + b.y}; }
__host__ __device__ inline zd operator-(zd a, zd b) { return {a.x - b.x, a.y - b.y}; }
__host__ __device__ inline zd operator*(zd a, zd b) { return {a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x}; }
__host__ __device__ inline zd conjz(zd a) { return {a.x, -a.y}; }
__host__ __device__ inline double conjz(double a) { return a; }
__host__ __device__ inline zd& operator+=(zd& a, zd b) { a.x += b.x; a.y += b.y; return a; }
__host__ __device__ inline void fmaInto(double& acc, double a, double b) { acc = fma(a, b, acc); }
__host__ __device__ inline void fmaInto(zd& acc, zd a, zd b) {
  acc.x = fma(a.x, b.x, acc.x); acc.x = fma(-a.y, b.y, acc.x);
  acc.y = fma(a.x, b.y, acc.y); acc.y = fma(a.y, b.x, acc.y);
}
template <class T> __host__ __device__ inline T zeroOf();
template <> __host__ __device__ inline double zeroOf<double>() { return 0.0; }
template <> __host__ __device__ inline zd zeroOf<zd>() { return {0.0, 0.0}; }
template <class T> __host__ __device__ inline T scalarOf(const double s[2]);
template <> __host__ __device__ inline double scalarOf<double>(const double s[2]) { return s[0]; }
template <> __host__ __device__ inline zd scalarOf<zd>(const double s[2]) { return {s[0], s[1]}; }
__host__ __device__ inline bool isZero(double a) { return a == 0.0; }
__host__ __device__ inline bool isZero(zd a) { return a.x == 0.0 && a.y == 0.0; }
__host__ __device__ inline bool isOne(double a) { return a == 1.0; }
__host__ __device__ inline bool isOne(zd a) { return a.x == 1.0 && a.y == 0.0; }

// Column pointer table passed by value to kernels: views with arbitrary column lists cost
// nothing extra (MxMultiVector.cpp:29-44 semantics).
template <class T>
struct ColTable {
  T* p[MXG_MAX_COLS];
};

}  // namespace mxg

struct mxg_ctx {
  int device = 0;
  int numSMs = 148;
  cudaStream_t stream = nullptr;       // compute stream
  cudaStream_t commStream = nullptr;   // halo exchange stream
  cudaEvent_t evA = nullptr, evB = nullptr;
  cudaEvent_t timer[16] = {};          // user timing slots (created lazily)
  cudaEvent_t prof[10] = {};           // per-kernel profiling events
  bool profiling = false;              // inside mxg_crs_apply_timed: record phase events, do not capture a graph
  ncclComm_t comm = nullptr;
  int rank = 0, nranks = 1;
  double* dScratch = nullptr;          // reduction partials / small device results
  size_t scratchBytes = 0;
  double* dDense = nullptr;            // device copy of the small dense B of the update product (kDenseBBytes)
  double* hPinned = nullptr;           // pinned host staging for small results and dense B
  size_t pinnedBytes = 0;
  int64_t launches = 0;
  bool graphsOff = false;              // set when stream capture of the halo apply is unavailable
  int* hErr = nullptr;                 // mapped pinned error word written by device-side waits
  int* dErr = nullptr;
  long long haloTimeoutTicks = 0;      // device clock ticks a halo wait may spin (MXG_HALO_TIMEOUT_S; 0 = for ever)
  uint64_t randomEpoch = 0;            // advanced by mxg_ctx_random_epoch: successive MvRandom calls draw new numbers
  int64_t asmBytes = 0, asmPeak = 0;   // device bytes held by the operator-assembly executors (mxg_asm_memory)
};

struct mxg_map {
  mxg_ctx* ctx = nullptr;
  int64_t nGlobal = 0, nLocal = 0;      // size of the GID space / DOFs owned by this rank
  int64_t nMapGlobal = -1;             // DOFs in the map over all ranks (lazily all-reduced: mxg::mapGlobalCount)
  std::vector<int64_t> gids;           // host copy (ascending)
  int64_t* dGids = nullptr;            // device copy (RNG keys, halo plans); in DEVICE order when the map is ordered
  // Optional component-major device ordering (mxg_map_create_ordered): perm[device position] = reference local index,
  // inv = its inverse. Empty = device order is the reference order (ascending GID).
  std::vector<int32_t> perm, inv;
  int refs = 1;
};

struct MvStorage {
  mxg_ctx* ctx = nullptr;
  void* base = nullptr;
  size_t bytes = 0;
  ~MvStorage();
};

struct mxg_mv {
  mxg_map* map = nullptr;
  bool isComplex = false;
  int ncols = 0;
  int64_t ld = 0;                          // local length (scalars per column)
  std::shared_ptr<MvStorage> storage;      // shared with views
  std::vector<void*> col;                  // device pointer of each column
  std::vector<int> baseCol;                // column position in the underlying allocation
};

namespace mxg {
struct HaloPeer {
  int rank = -1;
  int64_t sendCount = 0, sendOffset = 0;  // entries per column; offset into the send index list
  int64_t recvCount = 0, recvStart = 0;   // segment of the ghost list owned by this peer
};
}  // namespace mxg

struct mxg_crs {
  mxg_ctx* ctx = nullptr;
  mxg_map *rowMap = nullptr, *domMap = nullptr;
  bool isComplex = false;
  int64_t nRows = 0, nLoc = 0, nnz = 0;
  int64_t gLo = 0, gHi = 0;
  // dictionary path
  int32_t* dRowPat = nullptr;
  int32_t* dPatOff = nullptr;
  void* dPat = nullptr;
  int64_t numPats = 0, dictRows = 0, patEntries = 0;
  // general path
  int64_t nGen = 0, ellEntries = 0;
  int32_t* dGenRow = nullptr;
  int32_t* dGenLen = nullptr;
  int64_t* dSlicePtr = nullptr;
  int32_t* dCol = nullptr;
  void* dVal = nullptr;
  // rows [intBegin, intEnd) need no ghost values; general rows genIntBegin..genIntEnd lie inside it
  int64_t intBegin = 0, intEnd = 0, genIntBegin = 0, genIntEnd = 0;
  int64_t ghostRows = 0;
  // halo plan
  std::vector<mxg::HaloPeer> peers;
  int32_t* dSendIdx = nullptr;
  int64_t sendTotal = 0;
  mutable void* dSendBuf = nullptr;
  mutable void* dGhost = nullptr;
  mutable int haloCols = 0;
  size_t deviceBytes = 0;
  // 1 / diagonal (0 where the diagonal is 0 or absent); only for square operators whose row
  // and domain maps coincide -- the smoothers of the multigrid cycle use it
  void* dInvDiag = nullptr;
  int ilv = 1;                         // dictionary kernel: thread -> row interleave (1 or 3)
  // windowed dictionary kernel (mxg_spmm_win.cuh): per-tile x windows staged in shared memory by 1-D TMA
  void* dWinTiles = nullptr;           // WinTile[winTiles]
  int winR = 0;                        // rows per tile (0 = windowed path off)
  int winIlv = 1;                      // thread -> row assignment inside a tile (1 or 3)
  int winMaxVec = 1;                   // widest block the windowed kernel takes (wider blocks: gather kernels)
  int64_t winTiles = 0, winValid = 0;  // tiles / tiles served from shared memory
  int64_t winBufElems = 0;             // largest window set of any tile (scalars)
  // captured CUDA graphs of the multi-rank apply (pack -> NCCL exchange || interior rows -> boundary rows),
  // keyed by the operand pointers; replaying one costs a single launch instead of ~10 enqueues
  struct GraphEntry {
    uint64_t key;
    cudaGraphExec_t exec;
    int launches;
  };
  mutable std::vector<GraphEntry> graphs;
  // Direct peer-memory halo exchange: the whole apply is one launch (k_apply_fused) whose pack blocks store boundary values
  // straight into the neighbour's ghost buffer over NVLink, followed by an epoch flag; no NCCL call per apply.
  struct P2P {
    bool on = false;
    unsigned long long hostEpoch = 0;       // exchanges enqueued so far
    int capCols = 0;
    void* ghost = nullptr;                  // [2][capCols][gTot] scalars, IPC-exported (double buffered by epoch parity)
    unsigned long long* flags = nullptr;    // [nranks] epochs written by the senders, IPC-exported
    unsigned int* done = nullptr;           // block-completion counter of the pack kernel
    void* dArgs = nullptr;                  // device copy of the peer tables (P2PArgs) for the single-launch kernel
    unsigned long long* trace = nullptr;    // %globaltimer marks of the fused apply (mxg_crs_trace), NULL = off
    int npeers = 0;
    int peerRank[8];
    void* peerGhost[8];
    unsigned long long* peerFlag[8];
    int64_t remoteStart[8], remoteGTot[8];
    std::vector<void*> opened;
  };
  mutable P2P p2p;
};

namespace mxg {
template <class T>
inline ColTable<T> tableOf(const mxg_mv* mv, int first = 0, int count = -1) {
  ColTable<T> t;
  if (count < 0) count = mv->ncols - first;
  for (int j = 0; j < count; ++j) t.p[j] = static_cast<T*>(mv->col[first + j]);
  return t;
}
int ensureScratch(mxg_ctx* ctx, size_t bytes);
int ensurePinned(mxg_ctx* ctx, size_t bytes);
// sum `count` doubles in ctx->dScratch over all ranks (no-op on one rank)
int allReduceScratch(mxg_ctx* ctx, size_t count);
// number of DOFs of the map over all ranks (collective on first use when the context has several ranks)
int mapGlobalCount(mxg_map* map, int64_t* out);
// fails when a device-side halo wait has recorded a dead neighbour rank
int checkHaloFault(const mxg_ctx* ctx, const char* where);
// Device layout builder (mxg_spmv.cu): rows of a CRS matrix that already sits in device memory -> operator. dRowptr
// points at the first row of rowMap and holds offsets into dCol / dVal; columns are positions in the column field's map,
// of which domMap owns [colBegin, colBegin + nLocal). colFieldGids: host copy of that field map.
int crsCreateFromDevice(mxg_map* rowMap, mxg_map* domMap, const int64_t* dRowptr, const int32_t* dCol, const void* dVal, int64_t colBegin,
                        int64_t colFieldSize, const int64_t* colFieldGids, int isComplex, int layout, mxg_crs** out);
inline int gridFor(const mxg_ctx* ctx, int64_t work, int block, int perSM) {
  int64_t need = (work + block - 1) / block;
  int64_t cap = int64_t(ctx->numSMs) * perSM;
  if (need < 1) need = 1;
  return int(need < cap ? need : cap);
}
}  // namespace mxg
