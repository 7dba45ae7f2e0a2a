// libmxgpu: sparse operator apply (K1/K2/K4/K16/K20 of SURVEY.md section 2.3).
//
// Device layout ("pattern-compressed sliced ELL"), built by mxg_crs_create (host CSR) and mxg_crs_create_from_dcsr (device CSR):
//
//  * Dictionary rows. On a Yee grid almost every row of an assembled operator repeats the
//    same stencil: identical values and identical column offsets relative to the row.
//    Each distinct (offsets, values) tuple is stored ONCE in a pattern table and a row keeps
//    only a 4-byte pattern id. The apply then streams 4 B/row of matrix data instead of
//    12 B/nnz; x is gathered through L1/L2 and y written once.
//  * General rows (cut-cell rows next to the PEC wall, anything irregular) are kept in
//    sliced ELL with slice height 32 (one warp per slice, column-major inside the slice so
//    value and index loads are fully coalesced).
//  * Column indices live in an "extended" local index space [-gLo, nLoc + gHi): negative
//    and >= nLoc entries address the ghost buffer that the halo exchange fills, so ghost
//    rows use the same kernels and the same pattern table as interior rows.
//
// Arithmetic: each row is accumulated in ascending column order with separately rounded
// multiply and add, i.e. exactly the sequence Epetra_CrsMatrix::Apply executes on the CPU
// (complex rows follow the reference's real 2N "K form" order, MxCrsMatrix.cpp:145-170), so
// y = A x is bit-identical to the reference path, not merely within 1e-12.
#include <algorithm>
#include <cstdlib>
#include <cstring>

#include "mxg_internal.h"
#include "mxg_ilv_model.h"
#include "mxg_order.h"
#include "mxg_spmm_win.cuh"
#include "mxg_scan.cuh"

using namespace mxg;

namespace {

constexpr int kBlock = 256;

template <class T>
struct PatEntry;
template <>
struct __align__(16) PatEntry<double> {
  double v;
  int32_t d;
  int32_t pad;
};
template <>
struct __align__(16) PatEntry<zd> {
  double vx, vy;
  int32_t d;
  int32_t pad[3];
};

using Peer = mxg::HaloPeer;

// ---- exact (unfused) accumulation --------------------------------------------------------
__device__ __forceinline__ void accum(double& acc, double v, double x) { acc = __dadd_rn(acc, __dmul_rn(v, x)); }
__device__ __forceinline__ void accum(zd& acc, zd v, zd x) {
  // K-form row order: (re,re) (re,im) / (im,re) (im,im) -- MxCrsMatrix.cpp:158-168
  acc.x = __dadd_rn(acc.x, __dmul_rn(v.x, x.x));
  acc.x = __dadd_rn(acc.x, __dmul_rn(-v.y, x.y));
  acc.y = __dadd_rn(acc.y, __dmul_rn(v.y, x.x));
  acc.y = __dadd_rn(acc.y, __dmul_rn(v.x, x.y));
}
__device__ __forceinline__ double entryVal(const PatEntry<double>& e) { return e.v; }
__device__ __forceinline__ zd entryVal(const PatEntry<zd>& e) { return {e.vx, e.vy}; }

template <class T>
struct XSource {
  ColTable<T> x;       // local part of each column
  const T* ghost;      // [col][gLo + gHi]
  int64_t nLoc, gLo, gTot;
};

template <class T, bool GHOST>
__device__ __forceinline__ T loadX(const XSource<T>& X, int j, int64_t e) {
  if (GHOST) {
    if (e < 0) return X.ghost[j * X.gTot + (e + X.gLo)];
    if (e >= X.nLoc) return X.ghost[j * X.gTot + (e - X.nLoc + X.gLo)];
  }
  return ldgT(X.x.p[j] + e);
}

template <class T>
struct Epilogue {
  T alpha, beta;
  int mode;  // 0: y = acc, 1: y = alpha*acc + beta*y
};
template <class T>
__device__ __forceinline__ void storeY(T* y, int64_t row, T acc, const Epilogue<T>& ep) {
  if (ep.mode == 0) y[row] = acc;
  else if (isZero(ep.beta)) y[row] = ep.alpha * acc;
  else y[row] = ep.alpha * acc + ep.beta * y[row];
}

// Dictionary rows: one thread per row, two pattern entries per trip (no padded loads: ncu shows
// the kernel bound by L1 data-pipe wavefronts, l1tex__data_pipe_lsu_wavefronts 93%, so every
// extra load costs time).
template <class T>
struct DictArgs {
  const int32_t* rowPat;
  const int32_t* patOff;
  const PatEntry<T>* pat;
};
template <class T>
struct SellArgs {
  const int32_t* genRow;
  const int32_t* genLen;
  const int64_t* slicePtr;
  const int32_t* col;
  const T* val;
};

template <class T, bool GHOST, int NV>
__device__ __forceinline__ void dictRow(int64_t row, const DictArgs<T>& D, const XSource<T>& X,
                                        const ColTable<T>& Y, int nvec, const Epilogue<T>& ep) {
  const int32_t p = D.rowPat[row];
  if (p < 0) return;
  const int32_t o = __ldg(D.patOff + p), oe = __ldg(D.patOff + p + 1);
  for (int j0 = 0; j0 < nvec; j0 += NV) {
    T acc[NV];
#pragma unroll
    for (int jj = 0; jj < NV; ++jj) acc[jj] = zeroOf<T>();
    int32_t q = o;
    for (; q + 1 < oe; q += 2) {
      const PatEntry<T> e0 = D.pat[q];
      const PatEntry<T> e1 = D.pat[q + 1];
      T x0[NV], x1[NV];
#pragma unroll
      for (int jj = 0; jj < NV; ++jj) {
        x0[jj] = loadX<T, GHOST>(X, min(j0 + jj, nvec - 1), row + e0.d);
        x1[jj] = loadX<T, GHOST>(X, min(j0 + jj, nvec - 1), row + e1.d);
      }
#pragma unroll
      for (int jj = 0; jj < NV; ++jj) accum(acc[jj], entryVal(e0), x0[jj]);
#pragma unroll
      for (int jj = 0; jj < NV; ++jj) accum(acc[jj], entryVal(e1), x1[jj]);
    }
    if (q < oe) {
      const PatEntry<T> e0 = D.pat[q];
#pragma unroll
      for (int jj = 0; jj < NV; ++jj) accum(acc[jj], entryVal(e0), loadX<T, GHOST>(X, min(j0 + jj, nvec - 1), row + e0.d));
    }
#pragma unroll
    for (int jj = 0; jj < NV; ++jj)
      if (NV == 1 || j0 + jj < nvec) storeY(Y.p[j0 + jj], row, acc[jj], ep);
  }
}

// General rows: sliced ELL, slice height 32, one thread per (compacted) row. The loop runs over
// the slice width (uniform across the warp); entries past a row's own length are zero-padding
// and are skipped in the accumulation, which keeps the result bit-exact.
constexpr int kUnroll = 4;
template <class T, bool GHOST, int NV>
__device__ __forceinline__ void sellRow(int64_t i, const SellArgs<T>& S, const XSource<T>& X, const ColTable<T>& Y, int nvec,
                                        const Epilogue<T>& ep) {
  const int64_t row = S.genRow[i];
  const int len = row < 0 ? 0 : S.genLen[i];
  const int64_t sp = S.slicePtr[i >> 5];
  const int width = int((S.slicePtr[(i >> 5) + 1] - sp) >> 5);
  const int64_t base = sp + (i & 31);
  for (int j0 = 0; j0 < nvec; j0 += NV) {
    T acc[NV];
#pragma unroll
    for (int jj = 0; jj < NV; ++jj) acc[jj] = zeroOf<T>();
    for (int k = 0; k < width; k += kUnroll) {
      int32_t c[kUnroll];
      T v[kUnroll];
      T xv[kUnroll][NV];
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) {
        const int64_t at = base + int64_t(min(k + u, width - 1)) * 32;
        c[u] = S.col[at];
        v[u] = S.val[at];
      }
#pragma unroll
      for (int u = 0; u < kUnroll; ++u)
#pragma unroll
        for (int jj = 0; jj < NV; ++jj)
          xv[u][jj] = loadX<T, GHOST>(X, min(j0 + jj, nvec - 1), c[u]);  // padding holds a valid index
#pragma unroll
      for (int u = 0; u < kUnroll; ++u)
        if (k + u < len) {
#pragma unroll
          for (int jj = 0; jj < NV; ++jj) accum(acc[jj], v[u], xv[u][jj]);
        }
    }
    if (row >= 0) {
#pragma unroll
      for (int jj = 0; jj < NV; ++jj)
        if (NV == 1 || j0 + jj < nvec) storeY(Y.p[j0 + jj], row, acc[jj], ep);
    }
  }
}

// Sliced-ELL row without the unrolled index / value arrays of sellRow (those cost the single-launch kernel 16 registers and
// one CTA per SM); used for the few cut-cell rows inside k_apply_fused only. Same arithmetic order, bit-identical.
template <class T, bool GHOST>
__device__ __forceinline__ void sellRowSimple(int64_t i, const SellArgs<T>& S, const XSource<T>& X, const ColTable<T>& Y, int nvec,
                                              const Epilogue<T>& ep) {
  const int64_t row = S.genRow[i];
  if (row < 0) return;
  const int len = S.genLen[i];
  const int64_t base = S.slicePtr[i >> 5] + (i & 31);
  for (int j = 0; j < nvec; ++j) {
    T acc = zeroOf<T>();
    for (int k = 0; k < len; ++k) accum(acc, S.val[base + int64_t(k) * 32], loadX<T, GHOST>(X, j, S.col[base + int64_t(k) * 32]));
    storeY(Y.p[j], row, acc, ep);
  }
}

template <class T, bool GHOST, int NV>
__global__ void __launch_bounds__(kBlock) k_spmm_dict(int64_t rowBegin, int64_t rowEnd, DictArgs<T> D,
                                                      XSource<T> X, ColTable<T> Y, int nvec, Epilogue<T> ep) {
  const int64_t row = rowBegin + blockIdx.x * int64_t(kBlock) + threadIdx.x;
  if (row < rowEnd) dictRow<T, GHOST, NV>(row, D, X, Y, nvec, ep);
}

// Same rows, different thread -> row assignment for maps whose DOFs come in component triples (GID = comp + 3 cell,
// the B/E fields): warp w of a 96-row tile takes rows tile + 3 lane + (w mod 3), i.e. 32 consecutive CELLS of ONE field
// component. All lanes then share one pattern (one broadcast wavefront per entry instead of ~3) and gather x from one
// neighbourhood instead of three. Chosen per matrix at build time (mxg_crs::ilv), see planKernels.
constexpr int kBlockIlv = 384;   // 4 tiles of 3 warps
template <class T, bool GHOST, int NV>
__global__ void __launch_bounds__(kBlockIlv) k_spmm_dict_ilv3(int64_t rowBegin, int64_t rowEnd, DictArgs<T> D,
                                                              XSource<T> X, ColTable<T> Y, int nvec, Epilogue<T> ep) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row = rowBegin + blockIdx.x * int64_t(kBlockIlv) + (warp / 3) * 96 + 3 * lane + (warp % 3);
  if (row < rowEnd) dictRow<T, GHOST, NV>(row, D, X, Y, nvec, ep);
}


// ---- windowed dictionary kernel (design notes: mxg_spmm_win.cuh) ------------------------------------------------------
// One CTA per tile of R = kWinThreads * RPT consecutive rows. Thread 0 arms an mbarrier and issues <= 3 bulk copies that
// bring the tile's x windows into shared memory; meanwhile every warp fetches the pattern ids of its rows and stages the
// pattern ENTRIES in a per-warp shared slot (the shared-memory carve-out leaves little L1, and a dependent global load per
// entry made the first version of this kernel latency-bound: ncu, profiles/README_r02.md). The inner loop then touches
// shared memory only: one broadcast 16-byte load per entry (value + offset) and one 8-byte gather per lane.
// ILV = 3: warp w of a 384-row sub-tile takes rows 3*lane + (w mod 3) of its 96-row group -- 32 consecutive cells of ONE
// field component, which share a pattern and read the window with stride 3 (no bank conflict). ILV = 1: lane = row.
// A block of vectors is processed column by column through the same window buffer; several resident CTAs per SM overlap
// one tile's copy with another's arithmetic.
template <class T>
__device__ __forceinline__ void winIssue(const WinTile& W, const T* __restrict__ xcol, T* buf, uint64_t* bar) {
  uint32_t bytes = 0;
#pragma unroll
  for (int sgi = 0; sgi < 3; ++sgi) bytes += uint32_t(W.segLen[sgi]) * uint32_t(sizeof(T));
  mbarExpectTx(bar, bytes);
  int off = 0;
#pragma unroll
  for (int sgi = 0; sgi < 3; ++sgi) {
    if (W.segLen[sgi] > 0) bulkLoad(buf + off, xcol + W.segLo[sgi], uint32_t(W.segLen[sgi]) * uint32_t(sizeof(T)), bar);
    off += W.segLen[sgi];
  }
}

constexpr int kWinSlot = 16;   // pattern entries a per-warp slot holds (longer / non-uniform rows read the table directly)

template <class T>
__device__ __forceinline__ PatEntry<T> ldEntry(const PatEntry<T>* p) {
  // one (two for complex) 16-byte load instead of separate value / offset loads
  PatEntry<T> e;
  const int4* s = reinterpret_cast<const int4*>(p);
  int4* d = reinterpret_cast<int4*>(&e);
#pragma unroll
  for (int i = 0; i < int(sizeof(PatEntry<T>) / 16); ++i) d[i] = s[i];
  return e;
}

struct WinShift {
  int32_t dLo, dHi, s0, s1, s2;
};
// one row: entries from `ent` (per-warp shared slot or the global pattern table), x from the shared windows; ascending
// column order with separately rounded multiply and add, as everywhere in this file
template <class T>
__device__ __forceinline__ T winRowDot(const PatEntry<T>* __restrict__ ent, int32_t len, int32_t r, const T* __restrict__ xs, const WinShift& w) {
  T acc = zeroOf<T>();
  int32_t q = 0;
  for (; q + 1 < len; q += 2) {
    const PatEntry<T> e0 = ldEntry<T>(ent + q);
    const PatEntry<T> e1 = ldEntry<T>(ent + q + 1);
    const T x0 = xs[r + e0.d + (e0.d < w.dLo ? w.s0 : (e0.d > w.dHi ? w.s2 : w.s1))];
    const T x1 = xs[r + e1.d + (e1.d < w.dLo ? w.s0 : (e1.d > w.dHi ? w.s2 : w.s1))];
    accum(acc, entryVal(e0), x0);
    accum(acc, entryVal(e1), x1);
  }
  if (q < len) {
    const PatEntry<T> e0 = ldEntry<T>(ent + q);
    accum(acc, entryVal(e0), xs[r + e0.d + (e0.d < w.dLo ? w.s0 : (e0.d > w.dHi ? w.s2 : w.s1))]);
  }
  return acc;
}

template <class T, int ILV, int RPT>
__global__ void __launch_bounds__(kWinThreads) k_spmm_win(int64_t rowBegin, int64_t rowEnd, int64_t tile0, DictArgs<T> D,
                                                          const WinTile* __restrict__ tiles, XSource<T> X, ColTable<T> Y, int nvec,
                                                          Epilogue<T> ep) {
  extern __shared__ __align__(128) unsigned char smemRaw[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smemRaw);
  WinTile* Ws = reinterpret_cast<WinTile*>(smemRaw + 64);
  PatEntry<T>* slots = reinterpret_cast<PatEntry<T>*>(smemRaw + 128);
  constexpr int kWarps = kWinThreads / 32;
  T* buf = reinterpret_cast<T*>(smemRaw + 128 + sizeof(PatEntry<T>) * kWarps * RPT * kWinSlot);
  constexpr int R = kWinThreads * RPT;
  const int64_t tile = tile0 + blockIdx.x;
  if (threadIdx.x == 0) {
    const int4* src = reinterpret_cast<const int4*>(tiles + tile);
    int4* dst = reinterpret_cast<int4*>(Ws);
#pragma unroll
    for (int i = 0; i < 4; ++i) dst[i] = __ldg(src + i);
    mbarInit(bar, 1);
    mbarFenceInit();
    if (Ws->valid) winIssue<T>(*Ws, X.x.p[0], buf, bar);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tOff = ILV == 3 ? (warp / 3) * 96 + 3 * lane + (warp % 3) : int(threadIdx.x);
  int64_t row[RPT];
  int32_t o[RPT], len[RPT];
  bool uni[RPT];
#pragma unroll
  for (int i = 0; i < RPT; ++i) {
    row[i] = tile * R + i * kWinThreads + tOff;
    int32_t p = -1;
    if (row[i] >= rowBegin && row[i] < rowEnd) p = D.rowPat[row[i]];
    o[i] = len[i] = 0;
    if (p >= 0) { o[i] = __ldg(D.patOff + p); len[i] = __ldg(D.patOff + p + 1) - o[i]; }
    // warp-uniform pattern (lanes without a dictionary row do not count): stage its entries once for the whole warp
    const int32_t pmax = __reduce_max_sync(0xffffffffu, p);
    uni[i] = __all_sync(0xffffffffu, p < 0 || p == pmax) && pmax >= 0;
    const int32_t oU = __shfl_sync(0xffffffffu, o[i], __ffs(__ballot_sync(0xffffffffu, p == pmax)) - 1);
    const int32_t lenU = __shfl_sync(0xffffffffu, len[i], __ffs(__ballot_sync(0xffffffffu, p == pmax)) - 1);
    uni[i] = uni[i] && lenU <= kWinSlot;
    if (uni[i] && lane < lenU) slots[(warp * RPT + i) * kWinSlot + lane] = ldEntry<T>(D.pat + oU + lane);
  }
  __syncthreads();
  if (!Ws->valid) {   // tile-uniform: gather path
#pragma unroll
    for (int i = 0; i < RPT; ++i)
      if (row[i] >= rowBegin && row[i] < rowEnd) dictRow<T, false, 1>(row[i], D, X, Y, nvec, ep);
    return;
  }
  const int32_t dLo = Ws->dLo, dHi = Ws->dHi, s0 = Ws->shift[0], s1 = Ws->shift[1], s2 = Ws->shift[2];
  for (int j = 0; j < nvec; ++j) {
    mbarWait(bar, j & 1);
    const T* __restrict__ xs = buf;
#pragma unroll
    for (int i = 0; i < RPT; ++i) {
      if (len[i] == 0) continue;
      const int32_t r = int32_t(row[i]);
      const WinShift ws{dLo, dHi, s0, s1, s2};
      const T acc = uni[i] ? winRowDot<T>(slots + (warp * RPT + i) * kWinSlot, len[i], r, xs, ws)
                           : winRowDot<T>(D.pat + o[i], len[i], r, xs, ws);
      storeY(Y.p[j], row[i], acc, ep);
    }
    if (j + 1 < nvec) {
      __syncthreads();   // everyone is done with the windows of vector j
      if (threadIdx.x == 0) winIssue<T>(*Ws, X.x.p[j + 1], buf, bar);
    }
  }
}

template <class T, bool GHOST, int NV>
__global__ void __launch_bounds__(kBlock) k_spmm_sell(int64_t genBegin, int64_t genEnd, SellArgs<T> S,
                                                      XSource<T> X, ColTable<T> Y, int nvec, Epilogue<T> ep) {
  // genBegin is always a multiple of 32, so slices stay warp-aligned
  const int64_t i = genBegin + blockIdx.x * int64_t(kBlock) + threadIdx.x;
  if (i < genEnd) sellRow<T, GHOST, NV>(i, S, X, Y, nvec, ep);
}

// Several row ranges (dictionary + sliced ELL, leading + trailing boundary) in ONE launch: for short
// ranges the launch latency costs more than the rows.
struct Segments {
  int64_t begin[4], end[4];   // 0,1: dictionary row ranges; 2,3: sliced-ELL (compacted) ranges
  int blockStart[5];          // first block of each segment
};
template <class T, bool GHOST, int NV>
__global__ void __launch_bounds__(kBlock) k_spmm_multi(Segments G, DictArgs<T> D, SellArgs<T> S,
                                                       XSource<T> X, ColTable<T> Y, int nvec, Epilogue<T> ep) {
  int seg = 0;
  while (seg < 3 && int(blockIdx.x) >= G.blockStart[seg + 1]) ++seg;
  const int64_t idx = G.begin[seg] + int64_t(int(blockIdx.x) - G.blockStart[seg]) * kBlock + threadIdx.x;
  if (idx >= G.end[seg]) return;
  if (seg < 2) dictRow<T, GHOST, NV>(idx, D, X, Y, nvec, ep);
  else sellRow<T, GHOST, NV>(idx, S, X, Y, nvec, ep);
}

// halo pack: sendBuf[col][i] = x_col[sendIdx[i]]
template <class T>
__global__ void __launch_bounds__(kBlock) k_pack(ColTable<T> x, const int32_t* __restrict__ idx, int64_t n, T* __restrict__ buf) {
  const T* __restrict__ c = x.p[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock)
    buf[blockIdx.y * n + i] = c[idx[i]];
}

#define LAUNCH_CHECK(ctx)         \
  do {                            \
    (ctx)->launches++;            \
    MXG_CUDA(cudaGetLastError()); \
  } while (0)

template <class T>
DictArgs<T> dictArgs(const mxg_crs* A) { return {A->dRowPat, A->dPatOff, static_cast<const PatEntry<T>*>(A->dPat)}; }
template <class T>
SellArgs<T> sellArgs(const mxg_crs* A) { return {A->dGenRow, A->dGenLen, A->dSlicePtr, A->dCol, static_cast<const T*>(A->dVal)}; }

template <class T, bool GHOST>
int launchSegments(const mxg_crs* A, const int64_t b[4], const int64_t e[4], const XSource<T>& X, const ColTable<T>& Y, int nvec,
                   const Epilogue<T>& ep, cudaStream_t st) {
  mxg_ctx* ctx = A->ctx;
  Segments G;
  int blocks = 0;
  for (int sgm = 0; sgm < 4; ++sgm) {
    G.begin[sgm] = b[sgm];
    G.end[sgm] = e[sgm] > b[sgm] ? e[sgm] : b[sgm];
    G.blockStart[sgm] = blocks;
    blocks += int((G.end[sgm] - G.begin[sgm] + kBlock - 1) / kBlock);
  }
  G.blockStart[4] = blocks;
  if (blocks == 0) return MXG_OK;
  const DictArgs<T> D = dictArgs<T>(A);
  const SellArgs<T> S = sellArgs<T>(A);
  if (nvec == 1) k_spmm_multi<T, GHOST, 1><<<blocks, kBlock, 0, st>>>(G, D, S, X, Y, nvec, ep);
  else if (nvec == 2) k_spmm_multi<T, GHOST, 2><<<blocks, kBlock, 0, st>>>(G, D, S, X, Y, nvec, ep);
  else k_spmm_multi<T, GHOST, 4><<<blocks, kBlock, 0, st>>>(G, D, S, X, Y, nvec, ep);
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}


// rows per thread of the windowed kernel (tile = kWinThreads * RPT rows)
template <class T> struct WinCfg;
template <> struct WinCfg<double> { static constexpr int RPT = 2; };
template <> struct WinCfg<zd> { static constexpr int RPT = 1; };
constexpr size_t kWinSmemMax = 200 * 1024;      // per CTA
constexpr size_t kWinBufBudget = 100 * 1024;    // one window set
template <class T>
constexpr size_t winSmemHeader() { return 128 + sizeof(PatEntry<T>) * (kWinThreads / 32) * WinCfg<T>::RPT * kWinSlot; }

template <class T>
int launchWin(const mxg_crs* A, int64_t rowBegin, int64_t rowEnd, const XSource<T>& X, const ColTable<T>& Y, int nvec,
              const Epilogue<T>& ep, cudaStream_t st) {
  mxg_ctx* ctx = A->ctx;
  constexpr int RPT = WinCfg<T>::RPT;
  const int R = A->winR;
  const int64_t tile0 = rowBegin / R, tiles = (rowEnd + R - 1) / R - tile0;
  const size_t smem = winSmemHeader<T>() + size_t(A->winBufElems) * sizeof(T);
  const DictArgs<T> D = dictArgs<T>(A);
  const WinTile* wt = static_cast<const WinTile*>(A->dWinTiles);
  static bool attrSet[2] = {false, false};
  if (A->winIlv == 3) {
    auto kern = k_spmm_win<T, 3, RPT>;
    if (!attrSet[0]) { MXG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kWinSmemMax))); attrSet[0] = true; }
    kern<<<unsigned(tiles), kWinThreads, smem, st>>>(rowBegin, rowEnd, tile0, D, wt, X, Y, nvec, ep);
  } else {
    auto kern = k_spmm_win<T, 1, RPT>;
    if (!attrSet[1]) { MXG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kWinSmemMax))); attrSet[1] = true; }
    kern<<<unsigned(tiles), kWinThreads, smem, st>>>(rowBegin, rowEnd, tile0, D, wt, X, Y, nvec, ep);
  }
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}

// marks: record the per-kernel events of mxg_crs_apply_timed (prof[1..3]) around the launches
template <class T, bool GHOST>
int launchRange(const mxg_crs* A, int64_t rowBegin, int64_t rowEnd, int64_t genBegin, int64_t genEnd, const XSource<T>& X,
                const ColTable<T>& Y, int nvec, const Epilogue<T>& ep, bool marks) {
  mxg_ctx* ctx = A->ctx;
  const cudaStream_t st = ctx->stream;
  // Two launches on purpose: a merged kernel carries the register footprint of the sliced-ELL path
  // (unrolled index/value arrays) and the lost occupancy costs the L1-bound dictionary rows ~35 %
  // (measured 0.406 ms vs 0.299 ms per apply on pillbox-256). Only the short boundary ranges use the
  // merged kernel (launchBoundary).
  if (marks) MXG_CUDA(cudaEventRecord(ctx->prof[1], st));
  // The windowed kernel wins for single vectors (0.232 vs 0.262 ms on pillbox-256); for blocks the gather kernels share
  // every pattern load between 4 vectors and stay ahead (profiles/README_r02.md), so they keep the block applies.
  if (A->dictRows > 0 && rowEnd > rowBegin && A->winR > 0 && nvec <= A->winMaxVec) {
    const int rc = launchWin<T>(A, rowBegin, rowEnd, X, Y, nvec, ep, st);
    if (rc) return rc;
  } else if (A->dictRows > 0 && rowEnd > rowBegin) {
    const DictArgs<T> D = dictArgs<T>(A);
    if (A->ilv == 3) {
      const int64_t blocks = (rowEnd - rowBegin + kBlockIlv - 1) / kBlockIlv;
      if (nvec == 1) k_spmm_dict_ilv3<T, GHOST, 1><<<blocks, kBlockIlv, 0, st>>>(rowBegin, rowEnd, D, X, Y, nvec, ep);
      else if (nvec == 2) k_spmm_dict_ilv3<T, GHOST, 2><<<blocks, kBlockIlv, 0, st>>>(rowBegin, rowEnd, D, X, Y, nvec, ep);
      else k_spmm_dict_ilv3<T, GHOST, 4><<<blocks, kBlockIlv, 0, st>>>(rowBegin, rowEnd, D, X, Y, nvec, ep);
    } else {
      const int64_t blocks = (rowEnd - rowBegin + kBlock - 1) / kBlock;
      if (nvec == 1) k_spmm_dict<T, GHOST, 1><<<blocks, kBlock, 0, st>>>(rowBegin, rowEnd, D, X, Y, nvec, ep);
      else if (nvec == 2) k_spmm_dict<T, GHOST, 2><<<blocks, kBlock, 0, st>>>(rowBegin, rowEnd, D, X, Y, nvec, ep);
      else k_spmm_dict<T, GHOST, 4><<<blocks, kBlock, 0, st>>>(rowBegin, rowEnd, D, X, Y, nvec, ep);
    }
    LAUNCH_CHECK(ctx);
  }
  if (marks) MXG_CUDA(cudaEventRecord(ctx->prof[2], st));
  if (genEnd > genBegin) {
    const int64_t blocks = (genEnd - genBegin + kBlock - 1) / kBlock;
    const SellArgs<T> S = sellArgs<T>(A);
    if (nvec == 1) k_spmm_sell<T, GHOST, 1><<<blocks, kBlock, 0, st>>>(genBegin, genEnd, S, X, Y, nvec, ep);
    else if (nvec == 2) k_spmm_sell<T, GHOST, 2><<<blocks, kBlock, 0, st>>>(genBegin, genEnd, S, X, Y, nvec, ep);
    else k_spmm_sell<T, GHOST, 4><<<blocks, kBlock, 0, st>>>(genBegin, genEnd, S, X, Y, nvec, ep);
    LAUNCH_CHECK(ctx);
  }
  if (marks) MXG_CUDA(cudaEventRecord(ctx->prof[3], st));
  return MXG_OK;
}

// leading + trailing boundary rows (dictionary and sliced ELL) in one launch on stream st
template <class T>
int launchBoundary(const mxg_crs* A, const XSource<T>& X, const ColTable<T>& Y, int nvec, const Epilogue<T>& ep, cudaStream_t st) {
  const int64_t b[4] = {0, A->intEnd, 0, A->genIntEnd};
  const int64_t e[4] = {A->dictRows > 0 ? A->intBegin : 0, A->dictRows > 0 ? A->nRows : A->intEnd, A->genIntBegin, A->nGen};
  return launchSegments<T, true>(A, b, e, X, Y, nvec, ep, st);
}

__host__ __device__ inline uint64_t mix64(uint64_t h, uint64_t v) {
  h ^= v + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2);
  h *= 0xBF58476D1CE4E5B9ull;
  return h ^ (h >> 29);
}

// ---- peer-memory halo exchange --------------------------------------------------------------
// peer tables of the single-launch kernel, uploaded once per operator (mxg_crs::P2P::dArgs)
struct P2PArgs {
  int n;
  void* ghost[8];
  unsigned long long* flag[8];
  int64_t sendOffset[8], sendCount[8], remoteStart[8], remoteGTot[8];
  int senderRank[8];
};
// the single launch serves this block: peer memory is set up and its ghost buffers are wide enough
bool peerLaunch(const mxg_crs* A, int nvec) { return A->p2p.on && nvec <= A->p2p.capCols; }

// ---- the whole multi-rank apply in ONE launch -------------------------------------------------------------------------------
// Round 1 replayed a five-node graph (pack -> flag -> wait kernel -> boundary rows || interior rows) and measured ~100 us per
// apply waiting on the neighbours at 8 GPUs for ~33 us of interior work (profiles/README_r01.md): every link of that chain
// is a kernel with a 5-10 us floor. Here the roles are block ranges of one grid, in scheduling order:
//   [pack]      lowest block ids, resident first: boundary values of x go straight into the neighbours' ghost buffers
//               (NVLink stores), the last pack block publishes the epoch flag there
//   [interior]  dictionary + sliced-ELL rows that need no ghost value
//   [boundary]  highest block ids: wait for the neighbours' flags (they were written at the START of the neighbours' kernels),
//               then the rows that read ghosts
// A boundary block only ever waits for pack blocks of OTHER GPUs, which precede everything else in their grids, so the wait
// cannot dead-lock. The epoch is a kernel argument (counted on the host, identical on all ranks), the ghost buffers are
// double buffered by its parity. Reference call: the Epetra_Import inside Epetra_CrsMatrix::Apply (MxCrsMatrix.cpp:347-353).
constexpr int kFusedBlock = 384;
struct FusedPlan {
  int nPack, nDict;                   // blocks per role; boundary blocks follow
  int64_t dictBegin, dictEnd;         // interior dictionary rows
  int64_t bnd0Begin, bnd0End, bnd1Begin, bnd1End;   // boundary dictionary rows before / after the interior range
  int bndBlocks0, bndBlocks1;
  int nSellInt;                       // blocks of interior sliced-ELL rows (they run before the dictionary rows)
  int64_t sellIntBegin, sellIntEnd, nGen;   // sliced-ELL rows (compacted index space): interior range / all
  int ilv;
  unsigned long long epoch;
  unsigned long long* trace;          // optional %globaltimer timeline (mxg_crs_trace): [2 role] = min start, [2 role + 1] = max end
};
__device__ __forceinline__ unsigned long long globalTimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// roles: 0 pack, 1 interior dictionary rows, 2 interior sliced-ELL rows, 3 boundary wait, 4 boundary rows
__device__ __forceinline__ void traceMark(unsigned long long* trace, int role, bool end) {
  if (trace && threadIdx.x == 0) {
    const unsigned long long t = globalTimer();
    if (end) atomicMax(trace + 2 * role + 1, t);
    else atomicMin(trace + 2 * role, t);
  }
}
template <class T, int NV>
__global__ void __launch_bounds__(kFusedBlock, (NV == 1 && sizeof(T) == 8) ? 5 : (NV <= 2 ? 4 : 3)) k_apply_fused(FusedPlan F, const P2PArgs* __restrict__ P, const int32_t* __restrict__ sendIdx,
                                                             int64_t sendTotal, unsigned int* done, int capCols,
                                                             DictArgs<T> D, SellArgs<T> S, XSource<T> X, ColTable<T> Y, int nvec,
                                                             Epilogue<T> ep, const unsigned long long* flags, int* err,
                                                             long long timeoutTicks) {
  // The peer tables live in GLOBAL memory (P): indexing a kernel-parameter array with a run-time index makes the compiler
  // copy it to local memory at kernel entry in EVERY thread; those 160 B of local stores per thread evicted the gather
  // lines from L1 and cost the interior role 2.3x (ncu: profiles/r02_ncu_fused_self.json).
  int b = blockIdx.x;
  if (b < F.nPack) {
    traceMark(F.trace, 0, false);
    const unsigned long long par = F.epoch & 1ull;
    const int np = P->n;
    const int64_t total = sendTotal * nvec;
    for (int64_t e = b * int64_t(kFusedBlock) + threadIdx.x; e < total; e += int64_t(F.nPack) * kFusedBlock) {
      const int j = int(e / sendTotal);
      const int64_t i = e - int64_t(j) * sendTotal;
      int k = 0;
      while (k + 1 < np && i >= P->sendOffset[k] + P->sendCount[k]) ++k;
      T* dst = static_cast<T*>(P->ghost[k]) + (int64_t(par) * capCols + j) * P->remoteGTot[k] + P->remoteStart[k] + (i - P->sendOffset[k]);
      *dst = X.x.p[j][sendIdx[i]];
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
      if (atomicAdd(done, 1u) == unsigned(F.nPack) - 1u) {
        *done = 0u;
        __threadfence_system();
        for (int k = 0; k < np; ++k) *reinterpret_cast<volatile unsigned long long*>(P->flag[k]) = F.epoch;
        __threadfence_system();
      }
    }
    traceMark(F.trace, 0, true);
    return;
  }
  b -= F.nPack;
  if (b < F.nSellInt) {   // interior cut-cell rows: latency-bound (one dependent gather per entry), so they start early
    traceMark(F.trace, 2, false);
    const int64_t i = F.sellIntBegin + b * int64_t(kFusedBlock) + threadIdx.x;
    if (i < F.sellIntEnd) sellRowSimple<T, false>(i, S, X, Y, nvec, ep);
    if (F.trace) { __syncthreads(); traceMark(F.trace, 2, true); }
    return;
  }
  b -= F.nSellInt;
  if (b < F.nDict) {
    traceMark(F.trace, 1, false);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t row = F.dictBegin + b * int64_t(kFusedBlock) + (F.ilv == 3 ? (warp / 3) * 96 + 3 * lane + (warp % 3) : int(threadIdx.x));
    if (row < F.dictEnd) dictRow<T, false, NV>(row, D, X, Y, nvec, ep);
    if (F.trace) { __syncthreads(); traceMark(F.trace, 1, true); }
    return;
  }
  b -= F.nDict;
  // boundary rows. A neighbour that never publishes this epoch means a dead or dead-locked rank. Continuing would compute
  // boundary rows from stale ghost values and return wrong numbers with a success code, so the wait records the fault in the
  // mapped error word and traps: every later call on the context fails loudly.
  traceMark(F.trace, 3, false);
  if (int(threadIdx.x) < P->n) {
    const volatile unsigned long long* f = flags + P->senderRank[threadIdx.x];
    const long long t0 = clock64();
    while (*f < F.epoch) {
      if (timeoutTicks > 0 && clock64() - t0 > timeoutTicks) {
        *err = 1;
        __threadfence_system();
        asm volatile("trap;");
      }
      __nanosleep(32);
    }
    __threadfence_system();
  }
  __syncthreads();
  traceMark(F.trace, 3, true);
  traceMark(F.trace, 4, false);
  // two dictionary segments (rows before and after the interior range), then the sliced-ELL rows that read ghosts
  if (b < F.bndBlocks0 + F.bndBlocks1) {
    const bool second = b >= F.bndBlocks0;
    const int64_t idx = (second ? F.bnd1Begin + int64_t(b - F.bndBlocks0) * kFusedBlock : F.bnd0Begin + int64_t(b) * kFusedBlock) + threadIdx.x;
    if (idx < (second ? F.bnd1End : F.bnd0End)) dictRow<T, true, NV>(idx, D, X, Y, nvec, ep);
  } else {   // boundary cut-cell rows: the compacted ranges before and after the interior one
    int64_t i = int64_t(b - F.bndBlocks0 - F.bndBlocks1) * kFusedBlock + threadIdx.x;
    if (i >= F.sellIntBegin) i += F.sellIntEnd - F.sellIntBegin;
    if (i < F.nGen) sellRowSimple<T, true>(i, S, X, Y, nvec, ep);
  }
  if (F.trace) { __syncthreads(); traceMark(F.trace, 4, true); }
}

template <class T>
int launchFused(const mxg_crs* A, XSource<T> X, const ColTable<T>& Y, int nvec, const Epilogue<T>& ep) {
  mxg_ctx* ctx = A->ctx;
  auto& q = A->p2p;
  if (!q.dArgs) {   // device copy of the (static) peer tables
    P2PArgs P;
    P.n = q.npeers;
    for (int k = 0; k < q.npeers; ++k) {
      P.ghost[k] = q.peerGhost[k];
      P.flag[k] = q.peerFlag[k];
      P.remoteStart[k] = q.remoteStart[k];
      P.remoteGTot[k] = q.remoteGTot[k];
      P.senderRank[k] = q.peerRank[k];
      for (const Peer& pr : A->peers)
        if (pr.rank == q.peerRank[k]) { P.sendOffset[k] = pr.sendOffset; P.sendCount[k] = pr.sendCount; }
    }
    MXG_CUDA(cudaMalloc(&q.dArgs, sizeof(P2PArgs)));
    MXG_CUDA(cudaMemcpyAsync(q.dArgs, &P, sizeof(P2PArgs), cudaMemcpyHostToDevice, ctx->stream));
    MXG_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  FusedPlan F;
  F.nPack = A->sendTotal == 0 ? 0 : int(std::min<int64_t>(std::max<int64_t>(1, (A->sendTotal * nvec + 2 * kFusedBlock - 1) / (2 * kFusedBlock)), ctx->numSMs));
  F.dictBegin = A->dictRows > 0 ? A->intBegin : 0;
  F.dictEnd = A->dictRows > 0 ? A->intEnd : 0;
  F.nDict = int((F.dictEnd - F.dictBegin + kFusedBlock - 1) / kFusedBlock);
  F.ilv = A->ilv;
  F.epoch = q.hostEpoch;
  F.trace = q.trace;
  F.bnd0Begin = 0;
  F.bnd0End = A->dictRows > 0 ? A->intBegin : 0;
  F.bnd1Begin = A->intEnd;
  F.bnd1End = A->dictRows > 0 ? A->nRows : A->intEnd;
  F.bndBlocks0 = int((F.bnd0End - F.bnd0Begin + kFusedBlock - 1) / kFusedBlock);
  F.bndBlocks1 = int((F.bnd1End - F.bnd1Begin + kFusedBlock - 1) / kFusedBlock);
  F.nGen = A->nGen;
  F.sellIntBegin = A->genIntBegin;
  F.sellIntEnd = A->genIntEnd;
  F.nSellInt = int((F.sellIntEnd - F.sellIntBegin + kFusedBlock - 1) / kFusedBlock);
  // the blocks after the interior rows are also what WAITS for the neighbours' flags: keep one even when nothing reads a ghost
  int sellBlocks = int((A->nGen - (F.sellIntEnd - F.sellIntBegin) + kFusedBlock - 1) / kFusedBlock);
  if (A->sendTotal > 0 && F.bndBlocks0 + F.bndBlocks1 + sellBlocks == 0) F.bndBlocks1 = 1;
  X.ghost = static_cast<const T*>(q.ghost) + int64_t(F.epoch & 1ull) * q.capCols * X.gTot;   // this epoch's half of the double buffer
  const int grid = F.nPack + F.nSellInt + F.nDict + F.bndBlocks0 + F.bndBlocks1 + sellBlocks;
  const DictArgs<T> D = dictArgs<T>(A);
  const SellArgs<T> S = sellArgs<T>(A);
  const P2PArgs* dP = static_cast<const P2PArgs*>(q.dArgs);
  if (grid > 0) {
    if (nvec == 1) k_apply_fused<T, 1><<<grid, kFusedBlock, 0, ctx->stream>>>(F, dP, A->dSendIdx, A->sendTotal, q.done, q.capCols, D, S, X, Y, nvec, ep, q.flags, ctx->dErr, ctx->haloTimeoutTicks);
    else if (nvec == 2) k_apply_fused<T, 2><<<grid, kFusedBlock, 0, ctx->stream>>>(F, dP, A->dSendIdx, A->sendTotal, q.done, q.capCols, D, S, X, Y, nvec, ep, q.flags, ctx->dErr, ctx->haloTimeoutTicks);
    else k_apply_fused<T, 4><<<grid, kFusedBlock, 0, ctx->stream>>>(F, dP, A->dSendIdx, A->sendTotal, q.done, q.capCols, D, S, X, Y, nvec, ep, q.flags, ctx->dErr, ctx->haloTimeoutTicks);
    LAUNCH_CHECK(ctx);
  }
  return MXG_OK;
}

// pack -> grouped ncclSend/ncclRecv on the communication stream || interior rows -> boundary rows
// marks: record the phase events of mxg_crs_apply_timed (prof[1..3], prof[5])
template <class T>
int haloSequence(const mxg_crs* A, const XSource<T>& X, const ColTable<T>& Y, int nvec, const Epilogue<T>& ep, bool marks) {
  mxg_ctx* ctx = A->ctx;
  constexpr int w = sizeof(T) / sizeof(double);
  const int64_t gTot = A->gLo + A->gHi;
  // 1. pack boundary values and start the exchange on the communication stream
  T* sendBuf = static_cast<T*>(A->dSendBuf);
  T* ghost = static_cast<T*>(A->dGhost);
  if (A->sendTotal > 0) {
    k_pack<T><<<dim3(gridFor(ctx, A->sendTotal, kBlock, 4), nvec), kBlock, 0, ctx->stream>>>(X.x, A->dSendIdx, A->sendTotal, sendBuf);
    LAUNCH_CHECK(ctx);
  }
  MXG_CUDA(cudaEventRecord(ctx->evA, ctx->stream));
  MXG_CUDA(cudaStreamWaitEvent(ctx->commStream, ctx->evA, 0));
  if (marks) MXG_CUDA(cudaEventRecord(ctx->prof[1], ctx->commStream));
  MXG_NCCL(ncclGroupStart());
  for (const Peer& p : A->peers)
    for (int j = 0; j < nvec; ++j) {
      if (p.sendCount > 0)
        MXG_NCCL(ncclSend(sendBuf + j * A->sendTotal + p.sendOffset, size_t(p.sendCount) * w, ncclDouble, p.rank, ctx->comm, ctx->commStream));
      if (p.recvCount > 0)
        MXG_NCCL(ncclRecv(ghost + j * gTot + p.recvStart, size_t(p.recvCount) * w, ncclDouble, p.rank, ctx->comm, ctx->commStream));
    }
  MXG_NCCL(ncclGroupEnd());
  if (marks) MXG_CUDA(cudaEventRecord(ctx->prof[2], ctx->commStream));
  // 2. boundary rows follow the receive ON THE COMMUNICATION STREAM, so exchange + boundary work
  //    overlap with the interior rows running on the compute stream (they write disjoint rows of y)
  int rc = launchBoundary<T>(A, X, Y, nvec, ep, ctx->commStream);
  if (rc) return rc;
  MXG_CUDA(cudaEventRecord(ctx->evB, ctx->commStream));
  if (marks) MXG_CUDA(cudaEventRecord(ctx->prof[3], ctx->commStream));
  // 3. rows that need no ghost values
  if (marks) MXG_CUDA(cudaEventRecord(ctx->prof[5], ctx->stream));
  rc = launchRange<T, false>(A, A->intBegin, A->intEnd, A->genIntBegin, A->genIntEnd, X, Y, nvec, ep, false);
  if (rc) return rc;
  MXG_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->evB, 0));
  return MXG_OK;
}

template <class T>
int applyImpl(const mxg_crs* A, const mxg_mv* x, mxg_mv* y, const Epilogue<T>& ep) {
  mxg_ctx* ctx = A->ctx;
  const int nvec = x->ncols;
  const int64_t gTot = A->gLo + A->gHi;
  const bool halo = ctx->nranks > 1 && (gTot > 0 || A->sendTotal > 0);
  const bool timed = ctx->profiling;
  MXG_REQUIRE(*ctx->hErr == 0, "mxg_crs_apply: a previous halo exchange timed out waiting for a neighbour rank");
  if (halo && A->haloCols < nvec && !peerLaunch(A, nvec)) {
    MXG_CUDA(cudaStreamSynchronize(ctx->stream));
    MXG_CUDA(cudaStreamSynchronize(ctx->commStream));
    if (A->dSendBuf) MXG_CUDA(cudaFree(A->dSendBuf));
    if (A->dGhost) MXG_CUDA(cudaFree(A->dGhost));
    A->dSendBuf = A->dGhost = nullptr;
    for (auto& g : A->graphs) cudaGraphExecDestroy(g.exec);
    A->graphs.clear();
    MXG_CUDA(cudaMalloc(&A->dSendBuf, std::max<size_t>(16, sizeof(T) * A->sendTotal * nvec)));
    MXG_CUDA(cudaMalloc(&A->dGhost, std::max<size_t>(16, sizeof(T) * gTot * nvec)));
    A->haloCols = nvec;
  }
  XSource<T> X;
  X.x = tableOf<T>(x);
  X.ghost = static_cast<const T*>(A->dGhost);
  X.nLoc = A->nLoc;
  X.gLo = A->gLo;
  X.gTot = gTot;
  ColTable<T> Y = tableOf<T>(y);
  if (!halo) {
    // MXG_FUSED_SELF=1 (profiling aid): run the single-launch kernel of the multi-rank path on one rank, with empty pack and
    // boundary roles, so that ncu can look at its interior role
    const bool fusedSelf = std::getenv("MXG_FUSED_SELF") != nullptr;
    if (fusedSelf && ctx->nranks == 1 && A->dictRows > 0) return launchFused<T>(A, X, Y, nvec, ep);
    return launchRange<T, false>(A, 0, A->nRows, 0, A->nGen, X, Y, nvec, ep, timed);
  }
  if (peerLaunch(A, nvec)) {
    ++A->p2p.hostEpoch;   // one epoch per exchange, identical on all ranks
    return launchFused<T>(A, X, Y, nvec, ep);
  }

  // The multi-rank apply is ~10 enqueues (pack, events, NCCL group, 2-6 kernels) for tens of
  // microseconds of GPU work, i.e. launch-bound. Capture it once per operand set and replay.
  if (!ctx->graphsOff && !timed) {
    uint64_t key = mix64(0xC0FFEEull, uint64_t(nvec));
    for (int j = 0; j < nvec; ++j) { key = mix64(key, uint64_t(x->col[j])); key = mix64(key, uint64_t(y->col[j])); }
    uint64_t epBits[(sizeof(Epilogue<T>) + 7) / 8] = {};
    std::memcpy(epBits, &ep, sizeof(ep));
    for (uint64_t b : epBits) key = mix64(key, b);
    for (const auto& g : A->graphs)
      if (g.key == key) {
        MXG_CUDA(cudaGraphLaunch(g.exec, ctx->stream));
        ctx->launches += g.launches;
        return MXG_OK;
      }
    const int64_t before = ctx->launches;
    cudaGraph_t graph = nullptr;
    if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeRelaxed) == cudaSuccess) {
      const int rcCap = haloSequence<T>(A, X, Y, nvec, ep, false);
      const cudaError_t endErr = cudaStreamEndCapture(ctx->stream, &graph);
      cudaGraphExec_t exec = nullptr;
      if (rcCap == MXG_OK && endErr == cudaSuccess && graph && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) {
        cudaGraphDestroy(graph);
        if (A->graphs.size() >= 32) { cudaGraphExecDestroy(A->graphs.front().exec); A->graphs.erase(A->graphs.begin()); }
        A->graphs.push_back({key, exec, int(ctx->launches - before)});
        MXG_CUDA(cudaGraphLaunch(exec, ctx->stream));
        return MXG_OK;
      }
      if (graph) cudaGraphDestroy(graph);
    }
    cudaGetLastError();          // clear the capture error and fall back to eager enqueues for good
    ctx->launches = before;
    ctx->graphsOff = true;
  }
  return haloSequence<T>(A, X, Y, nvec, ep, timed);
}

// ---- host-side layout construction --------------------------------------------------------

template <class P>
int uploadVec(const std::vector<P>& v, P** out, size_t* bytes, mxg_ctx* ctx) {
  *out = nullptr;
  const size_t n = std::max<size_t>(v.size(), 1);
  MXG_CUDA(cudaMalloc(out, n * sizeof(P)));
  if (!v.empty()) MXG_CUDA(cudaMemcpyAsync(*out, v.data(), v.size() * sizeof(P), cudaMemcpyHostToDevice, ctx->stream));
  MXG_CUDA(cudaStreamSynchronize(ctx->stream));
  *bytes += n * sizeof(P);
  return MXG_OK;
}

// small host-table all-gather through a device bounce buffer (setup only)
template <class P>
int allGatherHost(mxg_ctx* ctx, const P* mine, size_t count, std::vector<P>& all) {
  const int R = ctx->nranks;
  const size_t bytes = sizeof(P) * count;
  char* d = nullptr;
  MXG_CUDA(cudaMalloc(&d, bytes * (R + 1)));
  MXG_CUDA(cudaMemcpyAsync(d + bytes * R, mine, bytes, cudaMemcpyHostToDevice, ctx->stream));
  MXG_NCCL(ncclAllGather(d + bytes * R, d, bytes, ncclChar, ctx->comm, ctx->stream));
  all.resize(count * R);
  MXG_CUDA(cudaMemcpyAsync(all.data(), d, bytes * R, cudaMemcpyDeviceToHost, ctx->stream));
  MXG_CUDA(cudaStreamSynchronize(ctx->stream));
  MXG_CUDA(cudaFree(d));
  return MXG_OK;
}

// Peer-memory exchange setup (collective): export this rank's ghost buffer + flag array with CUDA IPC,
// open the neighbours'. Every rank takes the same decision (all or none), otherwise the exchange
// would mix protocols and dead-lock.
int setupP2P(mxg_crs* A, int64_t gTot) {
  mxg_ctx* ctx = A->ctx;
  const int R = ctx->nranks;
  auto& q = A->p2p;
  const size_t esz = A->isComplex ? 16 : 8;
  const char* env = std::getenv("MXG_HALO");
  bool eligible = !(env && std::strcmp(env, "nccl") == 0) && A->peers.size() <= 8 && R <= 64;
  for (const Peer& p : A->peers)
    if (!(p.sendCount > 0 && p.recvCount > 0)) eligible = false;   // the epoch handshake needs symmetric neighbours
  int cap = 16;
  if (const char* c = std::getenv("MXG_P2P_COLS")) cap = std::max(1, std::atoi(c));
  struct Handles { cudaIpcMemHandle_t ghost, flags; };
  Handles mineH;
  std::memset(&mineH, 0, sizeof(mineH));
  if (eligible) {
    const size_t gb = size_t(2) * cap * std::max<int64_t>(gTot, 1) * esz;
    bool ok = cudaMalloc(&q.ghost, gb) == cudaSuccess && cudaMalloc(&q.flags, sizeof(unsigned long long) * R) == cudaSuccess &&
              cudaMalloc(&q.done, sizeof(unsigned int)) == cudaSuccess;
    if (ok) {
      cudaMemsetAsync(q.ghost, 0, gb, ctx->stream);
      cudaMemsetAsync(q.flags, 0, sizeof(unsigned long long) * R, ctx->stream);
      cudaMemsetAsync(q.done, 0, sizeof(unsigned int), ctx->stream);
      cudaStreamSynchronize(ctx->stream);
      ok = cudaIpcGetMemHandle(&mineH.ghost, q.ghost) == cudaSuccess && cudaIpcGetMemHandle(&mineH.flags, q.flags) == cudaSuccess;
    }
    if (!ok) { cudaGetLastError(); eligible = false; }
  }
  std::vector<int64_t> mine(R + 2, -1), all;
  for (const Peer& p : A->peers) mine[p.rank] = p.recvStart;
  mine[R] = gTot;
  mine[R + 1] = eligible ? 1 : 0;
  int rc = allGatherHost(ctx, mine.data(), mine.size(), all);
  if (rc) return rc;
  std::vector<Handles> allH;
  rc = allGatherHost(ctx, &mineH, 1, allH);
  if (rc) return rc;
  bool everyone = true;
  for (int r = 0; r < R; ++r) everyone = everyone && all[size_t(r) * (R + 2) + R + 1] == 1;
  int64_t opened = everyone ? 1 : 0;
  if (everyone) {
    q.npeers = 0;
    for (const Peer& p : A->peers) {
      void *pg = nullptr, *pf = nullptr;
      if (cudaIpcOpenMemHandle(&pg, allH[p.rank].ghost, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
          cudaIpcOpenMemHandle(&pf, allH[p.rank].flags, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError();
        if (pg) q.opened.push_back(pg);
        opened = 0;
        break;
      }
      q.opened.push_back(pg);
      q.opened.push_back(pf);
      const int k = q.npeers++;
      q.peerRank[k] = p.rank;
      q.peerGhost[k] = pg;
      q.peerFlag[k] = static_cast<unsigned long long*>(pf) + ctx->rank;
      q.remoteStart[k] = all[size_t(p.rank) * (R + 2) + ctx->rank];
      q.remoteGTot[k] = all[size_t(p.rank) * (R + 2) + R];
    }
  }
  // agree on the outcome
  int64_t* dflag = nullptr;
  MXG_CUDA(cudaMalloc(&dflag, sizeof(int64_t)));
  MXG_CUDA(cudaMemcpyAsync(dflag, &opened, sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
  MXG_NCCL(ncclAllReduce(dflag, dflag, 1, ncclInt64, ncclMin, ctx->comm, ctx->stream));
  MXG_CUDA(cudaMemcpyAsync(&opened, dflag, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
  MXG_CUDA(cudaStreamSynchronize(ctx->stream));
  MXG_CUDA(cudaFree(dflag));
  q.capCols = cap;
  q.on = opened == 1 && (gTot > 0 || A->sendTotal > 0);
  return MXG_OK;
}

// Who owns which ghost: every rank publishes its ghost GID list, owners answer with send lists.
int planHalo(mxg_crs* A, const std::vector<int64_t>& ghosts, const std::vector<int32_t>& domLookup, int64_t domLo, int64_t domHi) {
  mxg_ctx* ctx = A->ctx;
  const int P = ctx->nranks;
  if (P == 1) return MXG_OK;
  MXG_REQUIRE(ctx->comm != nullptr, "mxg_crs_create: %d ranks but no communicator (call mxg_ctx_comm_init)", P);
  // counts
  int64_t* dCnt = nullptr;
  MXG_CUDA(cudaMalloc(&dCnt, sizeof(int64_t) * (P + 1)));
  const int64_t mine = int64_t(ghosts.size());
  MXG_CUDA(cudaMemcpyAsync(dCnt + P, &mine, sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
  MXG_NCCL(ncclAllGather(dCnt + P, dCnt, 1, ncclInt64, ctx->comm, ctx->stream));
  std::vector<int64_t> cnt(P);
  MXG_CUDA(cudaMemcpyAsync(cnt.data(), dCnt, sizeof(int64_t) * P, cudaMemcpyDeviceToHost, ctx->stream));
  MXG_CUDA(cudaStreamSynchronize(ctx->stream));
  MXG_CUDA(cudaFree(dCnt));
  int64_t maxCnt = 1;
  for (int64_t c : cnt) maxCnt = std::max(maxCnt, c);
  // lists (padded)
  int64_t* dLists = nullptr;
  MXG_CUDA(cudaMalloc(&dLists, sizeof(int64_t) * maxCnt * (P + 1)));
  std::vector<int64_t> padded(maxCnt, -1);
  std::copy(ghosts.begin(), ghosts.end(), padded.begin());
  MXG_CUDA(cudaMemcpyAsync(dLists + maxCnt * P, padded.data(), sizeof(int64_t) * maxCnt, cudaMemcpyHostToDevice, ctx->stream));
  MXG_NCCL(ncclAllGather(dLists + maxCnt * P, dLists, maxCnt, ncclInt64, ctx->comm, ctx->stream));
  std::vector<int64_t> all(size_t(maxCnt) * P);
  MXG_CUDA(cudaMemcpyAsync(all.data(), dLists, sizeof(int64_t) * maxCnt * P, cudaMemcpyDeviceToHost, ctx->stream));
  MXG_CUDA(cudaStreamSynchronize(ctx->stream));
  MXG_CUDA(cudaFree(dLists));
  // domain ranges of every rank (to find the owner of my ghosts)
  int64_t* dRange = nullptr;
  MXG_CUDA(cudaMalloc(&dRange, sizeof(int64_t) * 2 * (P + 1)));
  const int64_t myRange[2] = {domLo, domHi};
  MXG_CUDA(cudaMemcpyAsync(dRange + 2 * P, myRange, sizeof(myRange), cudaMemcpyHostToDevice, ctx->stream));
  MXG_NCCL(ncclAllGather(dRange + 2 * P, dRange, 2, ncclInt64, ctx->comm, ctx->stream));
  std::vector<int64_t> ranges(2 * P);
  MXG_CUDA(cudaMemcpyAsync(ranges.data(), dRange, sizeof(int64_t) * 2 * P, cudaMemcpyDeviceToHost, ctx->stream));
  MXG_CUDA(cudaStreamSynchronize(ctx->stream));
  MXG_CUDA(cudaFree(dRange));

  std::vector<int32_t> sendIdx;
  A->peers.clear();
  for (int q = 0; q < P; ++q) {
    if (q == ctx->rank) continue;
    Peer peer;
    peer.rank = q;
    // what q needs from me
    peer.sendOffset = int64_t(sendIdx.size());
    for (int64_t i = 0; i < cnt[q]; ++i) {
      const int64_t g = all[size_t(q) * maxCnt + i];
      if (g >= domLo && g <= domHi) {
        const int32_t l = domLookup[g];
        MXG_REQUIRE(l >= 0, "mxg_crs_create: rank %d asks for GID %lld which lies in rank %d's range but is not in its map",
                    q, (long long)g, ctx->rank);
        sendIdx.push_back(l);
      }
    }
    peer.sendCount = int64_t(sendIdx.size()) - peer.sendOffset;
    // what I need from q: contiguous segment of my sorted ghost list
    const int64_t qLo = ranges[2 * q], qHi = ranges[2 * q + 1];
    if (qLo <= qHi) {
      auto b = std::lower_bound(ghosts.begin(), ghosts.end(), qLo);
      auto e = std::upper_bound(ghosts.begin(), ghosts.end(), qHi);
      peer.recvStart = int64_t(b - ghosts.begin());
      peer.recvCount = int64_t(e - b);
    }
    if (peer.sendCount > 0 || peer.recvCount > 0) A->peers.push_back(peer);
  }
  int64_t covered = 0;
  for (const Peer& p : A->peers) covered += p.recvCount;
  MXG_REQUIRE(covered == int64_t(ghosts.size()), "mxg_crs_create: %lld ghost columns have no owner",
              (long long)(int64_t(ghosts.size()) - covered));
  A->sendTotal = int64_t(sendIdx.size());
  // per-column send buffers are [col][sendTotal]: offsets above are already relative to sendTotal
  int rcU = uploadVec(sendIdx, &A->dSendIdx, &A->deviceBytes, ctx);
  if (rcU) return rcU;
  return setupP2P(A, int64_t(ghosts.size()));
}

// Kernel plans that depend on the row -> pattern map: thread -> row interleave of the gather kernels and the x windows of
// the windowed kernel. The layout back end hands in host copies of the row -> pattern map and the pattern table.
template <class T>
int planKernels(mxg_crs* A, const std::vector<int32_t>& rowPat, const std::vector<int32_t>& patOff, const std::vector<PatEntry<T>>& pat) {
  mxg_ctx* ctx = A->ctx;
  const int64_t nRows = A->nRows, nLoc = A->nLoc;
  int rc = MXG_OK;
  // ---- thread -> row assignment of the dictionary kernel: plain, or stride-3 component interleave. Chosen by a
  // line-count model over sampled interior tiles (mxg_ilv_model.h, with the B200 measurements that calibrate it).
  // MXG_SPMV_ILV = 1 / 3 forces either.
  {
    const char* env = std::getenv("MXG_SPMV_ILV");
    const std::string mode = env ? env : "auto";
    A->ilv = 1;
    if (mode == "3") A->ilv = 3;
    else if (mode != "1" && A->dictRows > 0) {
      const PatEntry<T>* pe = pat.data();
      const mxg::IlvCost cost = mxg::ilvCostModel(rowPat.data(), patOff.data(), [pe](int32_t q) { return pe[q].d; }, A->intBegin,
                                                  A->intEnd, int(sizeof(T)), int(sizeof(PatEntry<T>)));
      if (mxg::ilvWins(cost)) A->ilv = 3;
    }
  }

  // ---- windowed dictionary kernel: per-tile x windows (mxg_spmm_win.cuh). MXG_SPMV_WIN=0 keeps the gather kernels.
  {
    const char* env = std::getenv("MXG_SPMV_WIN");
    const bool want = !(env && std::strcmp(env, "0") == 0);
    if (want && A->dictRows > 0 && nLoc + A->gLo + A->gHi < (int64_t(1) << 30)) {
      constexpr int R = kWinThreads * WinCfg<T>::RPT;
      constexpr int align = 16 / int(sizeof(T)) > 0 ? 16 / int(sizeof(T)) : 1;
      const PatEntry<T>* pe = pat.data();
      int64_t maxTotal = 0, valid = 0;
      std::vector<WinTile> tiles = planWinTiles(rowPat.data(), patOff.data(), A->numPats, [pe](int32_t q) { return int64_t(pe[q].d); }, nRows,
                                                nLoc, R, align, int64_t(std::min(kWinBufBudget, kWinSmemMax - winSmemHeader<T>()) / sizeof(T)), &maxTotal, &valid);
      if (valid > 0) {
        WinTile* dT = nullptr;
        if ((rc = uploadVec(tiles, &dT, &A->deviceBytes, ctx))) return rc;
        A->dWinTiles = dT;
        A->winR = R;
        A->winTiles = int64_t(tiles.size());
        A->winValid = valid;
        A->winBufElems = maxTotal;
        A->winMaxVec = 1;
        if (const char* mv = std::getenv("MXG_WIN_MAXVEC")) A->winMaxVec = std::atoi(mv);
        // thread -> row assignment: component triples (GID = comp + 3 cell) share patterns at distance 3, scalar fields at 1
        int64_t same1 = 0, same3 = 0;
        for (int64_t r = 0; r + 3 < nRows; ++r) {
          if (rowPat[r] < 0) continue;
          same1 += rowPat[r] == rowPat[r + 1];
          same3 += rowPat[r] == rowPat[r + 3];
        }
        A->winIlv = same3 > same1 ? 3 : 1;
        if (const char* iv = std::getenv("MXG_SPMV_ILV")) {
          if (std::strcmp(iv, "1") == 0) A->winIlv = 1;
          if (std::strcmp(iv, "3") == 0) A->winIlv = 3;
        }
      }
    }
  }

  return rc;
}

// ---- layout construction ----------------------------------------------------------------------------------------------
// Two front ends bring a rank's rows into extended local columns: buildImpl from host CSR with global column ids
// (mxg_crs_create), buildFromDeviceImpl from CRS rows that already sit in device memory (the operator assembly, mxg_asm.cu).
// One back end, layoutFromDeviceRows, lays those rows out: the pattern dictionary (a device hash table), sliced ELL and the
// inverse diagonal are kernels; the host keeps what is small or collective -- pattern ordering (a few thousand
// candidates), the halo plan and the tile planner on a downloaded row -> pattern map.
struct Scratch {
  std::vector<void*> p;
  ~Scratch() { for (void* q : p) if (q) cudaFree(q); }
  template <class U>
  U* get(int64_t n) {
    void* q = nullptr;
    if (cudaMalloc(&q, size_t(n > 0 ? n : 1) * sizeof(U)) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    p.push_back(q);
    return static_cast<U*>(q);
  }
};

constexpr unsigned long long kLbEmpty = 0xFFFFFFFFFFFFFFFFull;

__global__ void k_lb_mark_ghosts(const int32_t* __restrict__ col, int64_t cnt, int64_t c0, int64_t c1, int32_t* __restrict__ flag) {
  for (int64_t q = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; q < cnt; q += int64_t(gridDim.x) * blockDim.x) {
    const int64_t l = col[q];
    if (l < c0 || l >= c1) flag[l] = 1;
  }
}
__global__ void k_lb_compact(const int32_t* __restrict__ flag, const int64_t* __restrict__ off, int64_t n, int32_t* __restrict__ list) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    if (flag[i]) list[off[i]] = int32_t(i);
}
// extended local column of every entry (owned: 0 .. nLoc-1; ghosts below / above the owned range: negative / >= nLoc)
__global__ void k_lb_ext(const int64_t* __restrict__ rp, const int32_t* __restrict__ colG, int64_t nRows, int64_t base, int64_t c0,
                         int64_t c1, int64_t nLoc, int64_t gLo, const int64_t* __restrict__ ghostOff, int32_t* __restrict__ ext,
                         uint8_t* __restrict__ needs, int* __restrict__ err) {
  for (int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; r < nRows; r += int64_t(gridDim.x) * blockDim.x) {
    bool ghost = false;
    for (int64_t q = rp[r]; q < rp[r + 1]; ++q) {
      const int64_t l = colG[q];
      int32_t e;
      if (l >= c0 && l < c1) e = int32_t(l - c0);
      else if (ghostOff) {
        const int64_t pos = ghostOff[l];
        e = pos < gLo ? int32_t(pos - gLo) : int32_t(nLoc + (pos - gLo));
        ghost = true;
      } else { *err = 1; e = 0; }
      ext[q - base] = e;
    }
    if (needs) needs[r] = ghost ? 1 : 0;
  }
}

template <class T>
__device__ __forceinline__ uint64_t lbRowHash(const int64_t* rp, const int32_t* ext, const T* valG, int64_t base, int64_t r) {
  constexpr int w = sizeof(T) / sizeof(double);
  const int64_t b = rp[r], e = rp[r + 1];
  uint64_t h = mix64(0x1234567ull, uint64_t(e - b));
  for (int64_t q = b; q < e; ++q) {
    h = mix64(h, uint64_t(int64_t(ext[q - base]) - r));
    const uint64_t* bits = reinterpret_cast<const uint64_t*>(valG + q);
    for (int t = 0; t < w; ++t) h = mix64(h, bits[t]);
  }
  return h == kLbEmpty ? h ^ 1ull : h;
}
template <class T>
__device__ __forceinline__ bool lbSameRow(const int64_t* rp, const int32_t* ext, const T* valG, int64_t base, int64_t a, int64_t b) {
  constexpr int w = sizeof(T) / sizeof(double);
  const int64_t la = rp[a + 1] - rp[a];
  if (la != rp[b + 1] - rp[b]) return false;
  for (int64_t k = 0; k < la; ++k) {
    const int64_t qa = rp[a] + k, qb = rp[b] + k;
    if (int64_t(ext[qa - base]) - a != int64_t(ext[qb - base]) - b) return false;
    const uint64_t* va = reinterpret_cast<const uint64_t*>(valG + qa);
    const uint64_t* vb = reinterpret_cast<const uint64_t*>(valG + qb);
    for (int t = 0; t < w; ++t)
      if (va[t] != vb[t]) return false;
  }
  return true;
}
// rows -> hash-table slots (open addressing, linear probing); the representative of a slot is its first row
template <class T>
__global__ void k_lb_hash_insert(const int64_t* __restrict__ rp, const int32_t* __restrict__ ext, const T* __restrict__ valG, int64_t base,
                                 int64_t nRows, unsigned long long* __restrict__ keys, int32_t* __restrict__ rep, int32_t* __restrict__ count,
                                 int32_t* __restrict__ rowSlot, uint64_t mask) {
  for (int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; r < nRows; r += int64_t(gridDim.x) * blockDim.x) {
    if (rp[r + 1] == rp[r]) { rowSlot[r] = -1; continue; }        // empty rows go to the general path (y = 0)
    const unsigned long long h = lbRowHash<T>(rp, ext, valG, base, r);
    uint64_t slot = (h * 0x9E3779B97F4A7C15ull >> 20) & mask;
    for (;;) {
      const unsigned long long old = atomicCAS(keys + slot, kLbEmpty, h);
      if (old == kLbEmpty || old == h) break;
      slot = (slot + 1) & mask;
    }
    atomicMin(rep + slot, int32_t(r));
    atomicAdd(count + slot, 1);
    rowSlot[r] = int32_t(slot);
  }
}
// a 64-bit collision (different rows, same hash) sends the later row to the general path
template <class T>
__global__ void k_lb_verify(const int64_t* __restrict__ rp, const int32_t* __restrict__ ext, const T* __restrict__ valG, int64_t base,
                            int64_t nRows, const int32_t* __restrict__ rep, int32_t* __restrict__ count, int32_t* __restrict__ rowSlot) {
  for (int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; r < nRows; r += int64_t(gridDim.x) * blockDim.x) {
    const int32_t s = rowSlot[r];
    if (s < 0) continue;
    const int64_t lead = rep[s];
    if (lead != r && !lbSameRow<T>(rp, ext, valG, base, lead, r)) {
      rowSlot[r] = -1;
      atomicSub(count + s, 1);
    }
  }
}
__global__ void k_lb_occupied(const unsigned long long* __restrict__ keys, int64_t n, int32_t* __restrict__ flag) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    flag[i] = keys[i] != kLbEmpty ? 1 : 0;
}
__global__ void k_lb_cands(const int32_t* __restrict__ flag, const int64_t* __restrict__ off, int64_t n, const int32_t* __restrict__ rep,
                           const int32_t* __restrict__ count, const int64_t* __restrict__ rp, int32_t* __restrict__ candRep,
                           int32_t* __restrict__ candCount, int32_t* __restrict__ candLen) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    if (flag[i]) {
      const int64_t c = off[i];
      const int32_t r = rep[i];
      candRep[c] = r;
      candCount[c] = count[i];
      candLen[c] = int32_t(rp[r + 1] - rp[r]);
    }
}
__global__ void k_lb_row_pat(const int32_t* __restrict__ rowSlot, const int64_t* __restrict__ off, const int32_t* __restrict__ candPat,
                             int64_t nRows, int32_t* __restrict__ rowPat) {
  for (int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; r < nRows; r += int64_t(gridDim.x) * blockDim.x) {
    const int32_t s = rowSlot[r];
    rowPat[r] = s >= 0 ? candPat[off[s]] : -1;
  }
}
__device__ __forceinline__ void lbStoreEntry(PatEntry<double>* e, double v, int32_t d) { e->v = v; e->d = d; e->pad = 0; }
__device__ __forceinline__ void lbStoreEntry(PatEntry<zd>* e, zd v, int32_t d) {
  e->vx = v.x; e->vy = v.y; e->d = d; e->pad[0] = e->pad[1] = e->pad[2] = 0;
}
template <class T>
__global__ void k_lb_fill_pat(int64_t numPats, const int32_t* __restrict__ patRep, const int32_t* __restrict__ patOff,
                              const int64_t* __restrict__ rp, const int32_t* __restrict__ ext, const T* __restrict__ valG, int64_t base,
                              PatEntry<T>* __restrict__ pat) {
  for (int64_t p = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; p < numPats; p += int64_t(gridDim.x) * blockDim.x) {
    const int64_t r = patRep[p];
    const int64_t b = rp[r], n = rp[r + 1] - b;
    for (int64_t k = 0; k < n; ++k) lbStoreEntry(pat + patOff[p] + k, valG[b + k], int32_t(int64_t(ext[b + k - base]) - r));
  }
}
__global__ void k_lb_is_gen(const int32_t* __restrict__ rowPat, int64_t nRows, int32_t* __restrict__ flag) {
  for (int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; r < nRows; r += int64_t(gridDim.x) * blockDim.x)
    flag[r] = rowPat[r] < 0 ? 1 : 0;
}
// general rows in three classes (leading boundary, interior, trailing boundary), each padded to whole slices
__global__ void k_lb_gen_rows(const int32_t* __restrict__ flag, const int64_t* __restrict__ off, const int64_t* __restrict__ rp, int64_t nRows,
                              int64_t intBegin, int64_t intEnd, int64_t off0, int64_t off1, int64_t base1, int64_t base2,
                              int32_t* __restrict__ genRow, int32_t* __restrict__ genLen) {
  for (int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; r < nRows; r += int64_t(gridDim.x) * blockDim.x) {
    if (!flag[r]) continue;
    int64_t pos;
    if (r < intBegin) pos = off[r];
    else if (r < intEnd) pos = base1 + (off[r] - off0);
    else pos = base2 + (off[r] - off1);
    genRow[pos] = int32_t(r);
    genLen[pos] = int32_t(rp[r + 1] - rp[r]);
  }
}
__global__ void k_lb_slice_width(const int32_t* __restrict__ genLen, int64_t nSlices, int32_t* __restrict__ w) {
  for (int64_t s = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; s < nSlices; s += int64_t(gridDim.x) * blockDim.x) {
    int32_t m = 0;
    for (int l = 0; l < 32; ++l) m = max(m, genLen[s * 32 + l]);
    w[s] = m;
  }
}
__global__ void k_lb_times32(int64_t* __restrict__ p, int64_t n) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) p[i] *= 32;
}
// one warp per slice: lane l owns row l of the slice; padding entries point at a column a real entry of the slice uses
// (value 0), so the kernel may load through them unconditionally
template <class T>
__global__ void k_lb_fill_ell(const int32_t* __restrict__ genRow, const int32_t* __restrict__ genLen, const int64_t* __restrict__ slicePtr,
                              const int64_t* __restrict__ rp, const int32_t* __restrict__ ext, const T* __restrict__ valG, int64_t base,
                              int64_t nSlices, int32_t* __restrict__ ellCol, T* __restrict__ ellVal) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5, nWarps = (int64_t(gridDim.x) * blockDim.x) >> 5;
  for (int64_t s = warp; s < nSlices; s += nWarps) {
    const int64_t i = s * 32 + lane;
    const int64_t row = genRow[i];
    const int32_t len = genLen[i];
    const int64_t b = row >= 0 ? rp[row] : 0;
    const bool real = row >= 0 && len > 0;
    const unsigned have = __ballot_sync(0xffffffffu, real);
    int32_t fallback = real ? ext[b - base] : 0;
    fallback = have ? __shfl_sync(0xffffffffu, fallback, __ffs(have) - 1) : 0;
    const int64_t p0 = slicePtr[s];
    const int32_t width = int32_t((slicePtr[s + 1] - p0) >> 5);
    for (int32_t k = 0; k < width; ++k) {
      const bool on = row >= 0 && k < len;
      ellCol[p0 + int64_t(k) * 32 + lane] = on ? ext[b + k - base] : fallback;
      ellVal[p0 + int64_t(k) * 32 + lane] = on ? valG[b + k] : zeroOf<T>();
    }
  }
}
__device__ __forceinline__ double lbInverse(double d) { return 1.0 / d; }
__device__ __forceinline__ zd lbInverse(zd d) {
  // two roundings, no FMA contraction: this pins the bits of the inverse diagonal, and so of every multigrid result
  const double m2 = __dadd_rn(__dmul_rn(d.x, d.x), __dmul_rn(d.y, d.y));
  return {d.x / m2, -d.y / m2};
}
template <class T>
__global__ void k_lb_inv_diag(const int64_t* __restrict__ rp, const int32_t* __restrict__ ext, const T* __restrict__ valG, int64_t base,
                              int64_t nRows, T* __restrict__ inv) {
  for (int64_t r = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; r < nRows; r += int64_t(gridDim.x) * blockDim.x) {
    T out = zeroOf<T>();
    for (int64_t q = rp[r]; q < rp[r + 1]; ++q)
      if (ext[q - base] == r) {
        const T d = valG[q];
        out = isZero(d) ? zeroOf<T>() : lbInverse(d);      // rows are merged: at most one matching entry
      }
    inv[r] = out;
  }
}

inline unsigned lbGrid(int64_t n, int block = 256) {
  const int64_t b = (n + block - 1) / block;
  return unsigned(std::max<int64_t>(1, std::min<int64_t>(b, int64_t(1) << 20)));
}
// scratch buffer from the enclosing `tmp`; a failure names the entry point `fn`
#define MXG_LB_ALLOC(var, type, count)                                                          \
  type* var = tmp.get<type>(count);                                                             \
  MXG_REQUIRE(var != nullptr, "%s: out of device memory (%s)", fn, #var)
#define MXG_LB_KEEP(dst, type, count)                                                           \
  do {                                                                                          \
    void* q_ = nullptr;                                                                         \
    MXG_CUDA(cudaMalloc(&q_, size_t((count) > 0 ? (count) : 1) * sizeof(type)));                \
    dst = static_cast<type*>(q_);                                                               \
    A->deviceBytes += size_t((count) > 0 ? (count) : 1) * sizeof(type);                         \
  } while (0)

// interior range = longest run of rows without ghost needs, and the number of rows that have them (no `needs`: none has)
void setInterior(mxg_crs* A, const std::vector<uint8_t>& needs) {
  const int64_t nRows = A->nRows;
  int64_t bestB = 0, bestE = 0, runB = 0;
  for (int64_t r = 0; r <= nRows; ++r)
    if (r == nRows || (!needs.empty() && needs[size_t(r)])) {
      if (r - runB > bestE - bestB) { bestB = runB; bestE = r; }
      runB = r + 1;
    }
  A->intBegin = bestB;
  A->intEnd = bestE;
  for (uint8_t n : needs) A->ghostRows += n;
}

// Back end of both front ends: pattern dictionary, kernel plans, sliced ELL and inverse diagonal from a rank's rows in
// device memory. Precondition: the maps, nRows / nLoc, gLo / gHi and the halo plan are set; intBegin / intEnd, ghostRows
// and nnz are set; dExt[q - base] holds the extended local column of entry q (dRp and dVal index entries from base); rows
// are merged, one entry per column. fn names the entry point in error messages.
template <class T>
int layoutFromDeviceRows(mxg_crs* A, const int64_t* dRp, const int32_t* dExt, const T* dVal, int64_t base, int layout, const char* fn) {
  mxg_ctx* ctx = A->ctx;
  cudaStream_t st = ctx->stream;
  const int64_t nRows = A->nRows, nLoc = A->nLoc;
  Scratch tmp;

  // ---- pattern dictionary
  std::vector<int32_t> rowPat(static_cast<size_t>(nRows), -1), patOff(1, 0);
  std::vector<PatEntry<T>> pat;
  MXG_LB_KEEP(A->dRowPat, int32_t, nRows);
  // Rectangular operators on two different maps (div, grad, curl, the multigrid transfers) have no translation-invariant
  // rows -- column minus row index drifts with the row -- so the dictionary pass would hash tens of millions of unique
  // rows for nothing: they go straight to sliced ELL.
  const bool sameMaps = A->rowMap == A->domMap || A->rowMap->gids == A->domMap->gids;
  bool haveDict = false;
  if (layout != 1 && sameMaps && nRows > 0) {
    int64_t tableSize = 1024;
    while (tableSize < 2 * nRows) tableSize <<= 1;
    MXG_LB_ALLOC(dKeys, unsigned long long, tableSize);
    MXG_LB_ALLOC(dRep, int32_t, tableSize);
    MXG_LB_ALLOC(dCount, int32_t, tableSize);
    MXG_LB_ALLOC(dRowSlot, int32_t, nRows);
    MXG_CUDA(cudaMemsetAsync(dKeys, 0xFF, size_t(tableSize) * sizeof(unsigned long long), st));
    MXG_CUDA(cudaMemsetAsync(dRep, 0x7F, size_t(tableSize) * sizeof(int32_t), st));
    MXG_CUDA(cudaMemsetAsync(dCount, 0, size_t(tableSize) * sizeof(int32_t), st));
    k_lb_hash_insert<T><<<lbGrid(nRows), 256, 0, st>>>(dRp, dExt, dVal, base, nRows, dKeys, dRep, dCount, dRowSlot, uint64_t(tableSize - 1));
    k_lb_verify<T><<<lbGrid(nRows), 256, 0, st>>>(dRp, dExt, dVal, base, nRows, dRep, dCount, dRowSlot);
    MXG_LB_ALLOC(dOcc, int32_t, tableSize);
    MXG_LB_ALLOC(dSlotOff, int64_t, tableSize + 1);
    k_lb_occupied<<<lbGrid(tableSize), 256, 0, st>>>(dKeys, tableSize, dOcc);
    int64_t nCand = 0;
    MXG_CUDA(exclusiveScan(ctx, dOcc, dSlotOff, tableSize, &nCand));
    ctx->launches += 3;
    MXG_LB_ALLOC(dCandRep, int32_t, nCand);
    MXG_LB_ALLOC(dCandCount, int32_t, nCand);
    MXG_LB_ALLOC(dCandLen, int32_t, nCand);
    MXG_LB_ALLOC(dCandPat, int32_t, nCand);
    k_lb_cands<<<lbGrid(tableSize), 256, 0, st>>>(dOcc, dSlotOff, tableSize, dRep, dCount, dRp, dCandRep, dCandCount, dCandLen);
    std::vector<int32_t> candRep(static_cast<size_t>(nCand), 0), candCount(static_cast<size_t>(nCand), 0), candLen(static_cast<size_t>(nCand), 0);
    MXG_CUDA(cudaMemcpyAsync(candRep.data(), dCandRep, size_t(nCand) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MXG_CUDA(cudaMemcpyAsync(candCount.data(), dCandCount, size_t(nCand) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MXG_CUDA(cudaMemcpyAsync(candLen.data(), dCandLen, size_t(nCand) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    MXG_CUDA(cudaStreamSynchronize(st));
    // pattern numbering: candidates in order of first appearance, most frequent first (stable; the leading ones ride in
    // the kernel parameter block), at least 4 rows
    std::vector<int32_t> byRow(static_cast<size_t>(nCand), 0);
    for (int64_t c = 0; c < nCand; ++c) byRow[size_t(c)] = int32_t(c);
    std::sort(byRow.begin(), byRow.end(), [&](int32_t a, int32_t b) { return candRep[size_t(a)] < candRep[size_t(b)]; });
    std::stable_sort(byRow.begin(), byRow.end(), [&](int32_t a, int32_t b) { return candCount[size_t(a)] > candCount[size_t(b)]; });
    const int minCount = 4;
    std::vector<int32_t> candPat(static_cast<size_t>(nCand), -1), patRep;
    for (int32_t c : byRow) {
      if (candCount[size_t(c)] < minCount) continue;
      candPat[size_t(c)] = int32_t(patRep.size());
      patRep.push_back(candRep[size_t(c)]);
      patOff.push_back(patOff.back() + candLen[size_t(c)]);
      A->dictRows += candCount[size_t(c)];
    }
    A->numPats = int64_t(patRep.size());
    A->patEntries = patOff.back();
    MXG_CUDA(cudaMemcpyAsync(dCandPat, candPat.data(), size_t(nCand) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    k_lb_row_pat<<<lbGrid(nRows), 256, 0, st>>>(dRowSlot, dSlotOff, dCandPat, nRows, A->dRowPat);
    MXG_LB_ALLOC(dPatRep, int32_t, A->numPats);
    MXG_LB_KEEP(A->dPatOff, int32_t, A->numPats + 1);
    PatEntry<T>* dPat = nullptr;
    MXG_LB_KEEP(dPat, PatEntry<T>, A->patEntries);
    A->dPat = dPat;
    MXG_CUDA(cudaMemcpyAsync(dPatRep, patRep.data(), patRep.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    MXG_CUDA(cudaMemcpyAsync(A->dPatOff, patOff.data(), patOff.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (A->numPats > 0) k_lb_fill_pat<T><<<lbGrid(A->numPats, 64), 64, 0, st>>>(A->numPats, dPatRep, A->dPatOff, dRp, dExt, dVal, base, dPat);
    ctx->launches += 3;
    pat.resize(static_cast<size_t>(A->patEntries));
    MXG_CUDA(cudaMemcpyAsync(rowPat.data(), A->dRowPat, size_t(nRows) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (A->patEntries > 0) MXG_CUDA(cudaMemcpyAsync(pat.data(), dPat, size_t(A->patEntries) * sizeof(PatEntry<T>), cudaMemcpyDeviceToHost, st));
    MXG_CUDA(cudaStreamSynchronize(st));      // candPat / patRep / patOff are host temporaries: done with them here
    haveDict = true;
  }
  if (!haveDict) {
    MXG_CUDA(cudaMemsetAsync(A->dRowPat, 0xFF, size_t(std::max<int64_t>(nRows, 1)) * sizeof(int32_t), st));
    MXG_LB_KEEP(A->dPatOff, int32_t, 1);
    MXG_CUDA(cudaMemsetAsync(A->dPatOff, 0, sizeof(int32_t), st));
    PatEntry<T>* dPat = nullptr;
    MXG_LB_KEEP(dPat, PatEntry<T>, 1);
    A->dPat = dPat;
  }
  // (A constant-bank copy of the most frequent patterns was tried and removed: 0.351 ms vs 0.305 ms per apply on
  // pillbox-256 -- a warp holds ~3 different patterns and divergent LDC replays cost more than L1 broadcast loads;
  // the 16 KB parameter block also lengthened every launch. profiles/README_r01.md.)
  int rc = planKernels<T>(A, rowPat, patOff, pat);
  if (rc) return rc;

  // ---- general rows in sliced ELL; the three row classes (leading boundary, interior, trailing boundary) each start on
  // a slice boundary so they can be launched separately
  MXG_LB_ALLOC(dIsGen, int32_t, nRows);
  MXG_LB_ALLOC(dGenOff, int64_t, nRows + 1);
  if (nRows > 0) k_lb_is_gen<<<lbGrid(nRows), 256, 0, st>>>(A->dRowPat, nRows, dIsGen);
  int64_t totalGen = 0;
  MXG_CUDA(exclusiveScan(ctx, dIsGen, dGenOff, nRows, &totalGen));
  int64_t offs[2] = {0, totalGen};
  MXG_CUDA(cudaMemcpyAsync(&offs[0], dGenOff + A->intBegin, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  MXG_CUDA(cudaMemcpyAsync(&offs[1], dGenOff + A->intEnd, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  MXG_CUDA(cudaStreamSynchronize(st));
  auto pad32 = [](int64_t v) { return (v + 31) / 32 * 32; };
  const int64_t n0 = offs[0], n1 = offs[1] - offs[0], n2 = totalGen - offs[1];
  A->genIntBegin = pad32(n0);
  A->genIntEnd = A->genIntBegin + pad32(n1);
  A->nGen = A->genIntEnd + pad32(n2);
  MXG_LB_KEEP(A->dGenRow, int32_t, A->nGen);
  MXG_LB_KEEP(A->dGenLen, int32_t, A->nGen);
  MXG_CUDA(cudaMemsetAsync(A->dGenRow, 0xFF, size_t(std::max<int64_t>(A->nGen, 1)) * sizeof(int32_t), st));
  MXG_CUDA(cudaMemsetAsync(A->dGenLen, 0, size_t(std::max<int64_t>(A->nGen, 1)) * sizeof(int32_t), st));
  if (nRows > 0)
    k_lb_gen_rows<<<lbGrid(nRows), 256, 0, st>>>(dIsGen, dGenOff, dRp, nRows, A->intBegin, A->intEnd, offs[0], offs[1], A->genIntBegin,
                                                 A->genIntEnd, A->dGenRow, A->dGenLen);
  const int64_t nSlices = A->nGen / 32;
  MXG_LB_ALLOC(dSliceW, int32_t, nSlices);
  MXG_LB_KEEP(A->dSlicePtr, int64_t, nSlices + 1);
  if (nSlices > 0) k_lb_slice_width<<<lbGrid(nSlices), 256, 0, st>>>(A->dGenLen, nSlices, dSliceW);
  int64_t totalW = 0;
  MXG_CUDA(exclusiveScan(ctx, dSliceW, A->dSlicePtr, nSlices, &totalW));
  k_lb_times32<<<lbGrid(nSlices + 1), 256, 0, st>>>(A->dSlicePtr, nSlices + 1);
  A->ellEntries = totalW * 32;
  MXG_LB_KEEP(A->dCol, int32_t, A->ellEntries);
  T* dEllVal = nullptr;
  MXG_LB_KEEP(dEllVal, T, A->ellEntries);
  A->dVal = dEllVal;
  if (nSlices > 0) k_lb_fill_ell<T><<<lbGrid(nSlices * 32), 256, 0, st>>>(A->dGenRow, A->dGenLen, A->dSlicePtr, dRp, dExt, dVal, base, nSlices, A->dCol, dEllVal);
  ctx->launches += 5;

  // ---- inverse diagonal for the smoothers (square operators on a single map only)
  if (nRows == nLoc && A->rowMap->gids == A->domMap->gids) {
    T* dInv = nullptr;
    void* q = nullptr;
    MXG_CUDA(cudaMalloc(&q, size_t(std::max<int64_t>(nRows, 1)) * sizeof(T)));
    dInv = static_cast<T*>(q);
    A->dInvDiag = dInv;
    if (nRows > 0) k_lb_inv_diag<T><<<lbGrid(nRows), 256, 0, st>>>(dRp, dExt, dVal, base, nRows, dInv);
    ctx->launches++;
  }
  MXG_CUDA(cudaGetLastError());
  MXG_CUDA(cudaStreamSynchronize(st));
  return MXG_OK;
}

// Host front end (mxg_crs_create): host CSR rows with global column ids.
template <class T>
int buildImpl(mxg_crs* A, const int64_t* rowptr, const int64_t* colGids, const double* valsIn, int layout) {
  const char* fn = "mxg_crs_create";
  mxg_ctx* ctx = A->ctx;
  const T* vals = reinterpret_cast<const T*>(valsIn);
  const int64_t nRows = A->nRows, nLoc = A->nLoc;
  const int64_t nnzIn = rowptr[nRows];
  const mxg_map* dom = A->domMap;
  MXG_REQUIRE(dom->nGlobal < (int64_t(1) << 31), "mxg_crs_create: global size must fit in 31 bits");

  // GID -> local id of the domain map
  std::vector<int32_t> lookup(size_t(dom->nGlobal), -1);
  for (int64_t i = 0; i < nLoc; ++i) lookup[dom->gids[i]] = int32_t(i);
  const int64_t domLo = nLoc ? dom->gids.front() : 0, domHi = nLoc ? dom->gids.back() : -1;

  // ghosts = referenced GIDs that are not local
  std::vector<int64_t> ghosts;
  for (int64_t q = 0; q < nnzIn; ++q) {
    const int64_t g = colGids[q];
    MXG_REQUIRE(g >= 0 && g < dom->nGlobal, "mxg_crs_create: column GID %lld out of range", (long long)g);
    if (lookup[g] < 0) ghosts.push_back(g);
  }
  std::sort(ghosts.begin(), ghosts.end());
  ghosts.erase(std::unique(ghosts.begin(), ghosts.end()), ghosts.end());
  MXG_REQUIRE(ghosts.empty() || ctx->nranks > 1, "mxg_crs_create: column GID %lld is not in the domain map",
              (long long)(ghosts.empty() ? 0 : ghosts[0]));
  A->gLo = int64_t(std::lower_bound(ghosts.begin(), ghosts.end(), domLo) - ghosts.begin());
  if (nLoc == 0) A->gLo = 0;
  A->gHi = int64_t(ghosts.size()) - A->gLo;
  int rc = planHalo(A, ghosts, lookup, domLo, domHi);
  if (rc) return rc;

  // extended local column index of every entry; rows sorted, duplicates merged
  std::vector<int64_t> rp(nRows + 1, 0);
  std::vector<int32_t> ext;
  std::vector<T> val;
  ext.reserve(nnzIn);
  val.reserve(nnzIn);
  std::vector<uint8_t> needsGhost(nRows, 0);
  std::vector<std::pair<int32_t, T>> rowBuf;
  for (int64_t r = 0; r < nRows; ++r) {
    rowBuf.clear();
    bool sorted = true;
    for (int64_t q = rowptr[r]; q < rowptr[r + 1]; ++q) {
      const int64_t g = colGids[q];
      int32_t e = lookup[g];
      if (e < 0) {
        const int64_t pos = std::lower_bound(ghosts.begin(), ghosts.end(), g) - ghosts.begin();
        e = pos < A->gLo ? int32_t(pos - A->gLo) : int32_t(nLoc + (pos - A->gLo));
        needsGhost[r] = 1;
      }
      if (!rowBuf.empty() && e <= rowBuf.back().first) sorted = false;
      rowBuf.emplace_back(e, vals[q]);
    }
    if (!sorted) {
      std::stable_sort(rowBuf.begin(), rowBuf.end(), [](auto& a, auto& b) { return a.first < b.first; });
      size_t o = 0;
      for (size_t i = 0; i < rowBuf.size();) {
        T s = rowBuf[i].second;
        size_t j = i + 1;
        while (j < rowBuf.size() && rowBuf[j].first == rowBuf[i].first) s = s + rowBuf[j++].second;
        rowBuf[o++] = {rowBuf[i].first, s};
        i = j;
      }
      rowBuf.resize(o);
    }
    for (auto& t : rowBuf) { ext.push_back(t.first); val.push_back(t.second); }
    rp[r + 1] = int64_t(ext.size());
  }
  A->nnz = int64_t(ext.size());
  // Ordered maps (mxg_map_create_ordered): rows move to their device positions and owned columns are translated; the
  // entry order inside a row stays the reference's ascending local column, so sums keep Epetra's order bit for bit.
  if (!A->rowMap->perm.empty() || !A->domMap->perm.empty()) {
    MXG_REQUIRE(ctx->nranks == 1 && ghosts.empty(), "mxg_crs_create: ordered maps are supported on single-rank contexts only");
    std::vector<int32_t> rowPerm = A->rowMap->perm, colInv = A->domMap->inv;
    if (rowPerm.empty()) { rowPerm.resize(size_t(nRows)); for (int64_t i = 0; i < nRows; ++i) rowPerm[size_t(i)] = int32_t(i); }
    if (colInv.empty()) { colInv.resize(size_t(nLoc)); for (int64_t i = 0; i < nLoc; ++i) colInv[size_t(i)] = int32_t(i); }
    std::vector<int64_t> rp2;
    std::vector<int32_t> ext2;
    std::vector<T> val2;
    try {
      mxg::permuteCsr(rp, ext, val, rowPerm, colInv, nLoc, rp2, ext2, val2);
    } catch (const std::exception& e) {   // nothing may unwind through the C boundary
      MXG_REQUIRE(false, "mxg_crs_create: %s", e.what());
    }
    rp.swap(rp2);
    ext.swap(ext2);
    val.swap(val2);
  }
  setInterior(A, needsGhost);

  // the merged rows go to the device for the common back end
  Scratch tmp;
  MXG_LB_ALLOC(dRp, int64_t, nRows + 1);
  MXG_LB_ALLOC(dExt, int32_t, A->nnz);
  MXG_LB_ALLOC(dVal, T, A->nnz);
  cudaStream_t st = ctx->stream;
  MXG_CUDA(cudaMemcpyAsync(dRp, rp.data(), rp.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  if (A->nnz > 0) {
    MXG_CUDA(cudaMemcpyAsync(dExt, ext.data(), ext.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    MXG_CUDA(cudaMemcpyAsync(dVal, val.data(), val.size() * sizeof(T), cudaMemcpyHostToDevice, st));
  }
  return layoutFromDeviceRows<T>(A, dRp, dExt, dVal, 0, layout, fn);
}

// Device front end (mxg_crs_create_from_dcsr): rows [base, base + nnz) of a device CRS whose columns are positions in
// the column field's map, of which this rank owns [c0, c0 + nLoc).
template <class T>
int buildFromDeviceImpl(mxg_crs* A, const int64_t* dRp, const int32_t* dColG, const void* dValRaw, int64_t c0, int64_t colFieldSize,
                        const int64_t* colFieldGids, int layout) {
  const char* fn = "mxg_crs_create_from_dcsr";
  mxg_ctx* ctx = A->ctx;
  cudaStream_t st = ctx->stream;
  const int64_t nRows = A->nRows, nLoc = A->nLoc, c1 = c0 + nLoc;
  const mxg_map* dom = A->domMap;
  MXG_REQUIRE(dom->nGlobal < (int64_t(1) << 31), "mxg_crs_create: global size must fit in 31 bits");
  Scratch tmp;
  int64_t ends[2] = {0, 0};
  MXG_CUDA(cudaMemcpyAsync(&ends[0], dRp, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  MXG_CUDA(cudaMemcpyAsync(&ends[1], dRp + nRows, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  MXG_CUDA(cudaStreamSynchronize(st));
  const int64_t base = ends[0], cnt = ends[1] - ends[0];
  A->nnz = cnt;
  const int64_t domLo = nLoc ? dom->gids.front() : 0, domHi = nLoc ? dom->gids.back() : -1;

  // ---- ghosts: referenced columns outside this rank's run of the column field map
  std::vector<int64_t> ghosts;
  int64_t* dGhostOff = nullptr;
  if (ctx->nranks > 1) {
    MXG_LB_ALLOC(dFlag, int32_t, colFieldSize);
    MXG_LB_ALLOC(dOff, int64_t, colFieldSize + 1);
    MXG_CUDA(cudaMemsetAsync(dFlag, 0, size_t(colFieldSize) * sizeof(int32_t), st));
    if (cnt > 0) k_lb_mark_ghosts<<<lbGrid(cnt), 256, 0, st>>>(dColG + base, cnt, c0, c1, dFlag);
    int64_t ng = 0;
    MXG_CUDA(exclusiveScan(ctx, dFlag, dOff, colFieldSize, &ng));
    if (ng > 0) {
      MXG_LB_ALLOC(dList, int32_t, ng);
      k_lb_compact<<<lbGrid(colFieldSize), 256, 0, st>>>(dFlag, dOff, colFieldSize, dList);
      std::vector<int32_t> list(static_cast<size_t>(ng), 0);
      MXG_CUDA(cudaMemcpyAsync(list.data(), dList, size_t(ng) * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
      MXG_CUDA(cudaStreamSynchronize(st));
      ghosts.resize(static_cast<size_t>(ng));
      for (int64_t i = 0; i < ng; ++i) ghosts[size_t(i)] = colFieldGids[list[size_t(i)]];   // ascending: the field map is
    }
    dGhostOff = dOff;
    ctx->launches += 2;
  }
  A->gLo = int64_t(std::lower_bound(ghosts.begin(), ghosts.end(), domLo) - ghosts.begin());
  if (nLoc == 0) A->gLo = 0;
  A->gHi = int64_t(ghosts.size()) - A->gLo;
  {
    std::vector<int32_t> lookup;
    if (ctx->nranks > 1) {
      lookup.assign(size_t(dom->nGlobal), -1);
      for (int64_t i = 0; i < nLoc; ++i) lookup[size_t(dom->gids[size_t(i)])] = int32_t(i);
    }
    const int rcH = planHalo(A, ghosts, lookup, domLo, domHi);
    if (rcH) return rcH;
  }

  // ---- extended local columns, rows that need ghost values
  MXG_LB_ALLOC(dExt, int32_t, cnt);
  MXG_LB_ALLOC(dErr, int, 1);
  uint8_t* dNeeds = nullptr;
  if (ctx->nranks > 1) { MXG_LB_ALLOC(needs_, uint8_t, nRows); dNeeds = needs_; }
  MXG_CUDA(cudaMemsetAsync(dErr, 0, sizeof(int), st));
  if (nRows > 0) k_lb_ext<<<lbGrid(nRows), 256, 0, st>>>(dRp, dColG, nRows, base, c0, c1, nLoc, A->gLo, dGhostOff, dExt, dNeeds, dErr);
  ctx->launches++;
  int hErr = 0;
  MXG_CUDA(cudaMemcpyAsync(&hErr, dErr, sizeof(int), cudaMemcpyDeviceToHost, st));
  std::vector<uint8_t> needs;
  if (dNeeds) {
    needs.resize(static_cast<size_t>(nRows));
    MXG_CUDA(cudaMemcpyAsync(needs.data(), dNeeds, size_t(nRows), cudaMemcpyDeviceToHost, st));
  }
  MXG_CUDA(cudaStreamSynchronize(st));
  MXG_REQUIRE(hErr == 0, "mxg_crs_create: a column is not in the domain map (single-rank context)");
  setInterior(A, needs);
  return layoutFromDeviceRows<T>(A, dRp, dExt, static_cast<const T*>(dValRaw), base, layout, fn);
}

// A new operator on (rowMap, domMap), laid out by `build`; released again when that fails.
template <class Build>
int crsCreate(mxg_map* rowMap, mxg_map* domMap, int isComplex, mxg_crs** out, Build build) {
  mxg_ctx* ctx = rowMap->ctx;
  MXG_CUDA(cudaSetDevice(ctx->device));
  mxg_crs* A = new mxg_crs;
  A->ctx = ctx;
  A->rowMap = rowMap;
  A->domMap = domMap;
  rowMap->refs++;
  domMap->refs++;
  A->isComplex = isComplex != 0;
  A->nRows = rowMap->nLocal;
  A->nLoc = domMap->nLocal;
  const int rc = build(A);
  if (rc) {
    mxg_crs_destroy(A);
    return rc;
  }
  *out = A;
  return MXG_OK;
}

}  // namespace

namespace mxg {

// rows [r0, r0 + rowMap->nLocal) of a device CRS (dRowptr points at row r0 and holds offsets into dCol / dVal; columns are
// positions in the column field's map, of which domMap owns [colBegin, colBegin + nLocal)) -> device operator
int crsCreateFromDevice(mxg_map* rowMap, mxg_map* domMap, const int64_t* dRowptr, const int32_t* dCol, const void* dVal, int64_t colBegin,
                        int64_t colFieldSize, const int64_t* colFieldGids, int isComplex, int layout, mxg_crs** out) {
  MXG_REQUIRE(rowMap && domMap && dRowptr && out, "mxg_crs_create_from_dcsr: NULL argument");
  MXG_REQUIRE(rowMap->ctx == domMap->ctx, "mxg_crs_create_from_dcsr: maps live on different contexts");
  MXG_REQUIRE(layout >= 0 && layout <= 1, "mxg_crs_create_from_dcsr: unknown layout %d", layout);
  MXG_REQUIRE(rowMap->perm.empty() && domMap->perm.empty(), "mxg_crs_create_from_dcsr: ordered maps are not supported by the device front end");
  return crsCreate(rowMap, domMap, isComplex, out, [&](mxg_crs* A) {
    return A->isComplex ? buildFromDeviceImpl<zd>(A, dRowptr, dCol, dVal, colBegin, colFieldSize, colFieldGids, layout)
                        : buildFromDeviceImpl<double>(A, dRowptr, dCol, dVal, colBegin, colFieldSize, colFieldGids, layout);
  });
}

}  // namespace mxg

extern "C" {

int mxg_crs_create_opts(mxg_map* row_map, mxg_map* domain_map, const int64_t* rowptr, const int64_t* col_gids,
                        const double* vals, int is_complex, int layout, mxg_crs** out) {
  MXG_REQUIRE(row_map && domain_map && rowptr && out, "mxg_crs_create: NULL argument");
  MXG_REQUIRE(row_map->ctx == domain_map->ctx, "mxg_crs_create: maps live on different contexts");
  MXG_REQUIRE(rowptr[0] == 0, "mxg_crs_create: rowptr[0] must be 0");
  const int64_t nnz = rowptr[row_map->nLocal];
  MXG_REQUIRE(nnz == 0 || (col_gids && vals), "mxg_crs_create: NULL column / value array");
  MXG_REQUIRE(layout >= 0 && layout <= 1, "mxg_crs_create: unknown layout %d", layout);
  return crsCreate(row_map, domain_map, is_complex, out, [&](mxg_crs* A) {
    return A->isComplex ? buildImpl<zd>(A, rowptr, col_gids, vals, layout) : buildImpl<double>(A, rowptr, col_gids, vals, layout);
  });
}

int mxg_crs_create(mxg_map* row_map, mxg_map* domain_map, const int64_t* rowptr, const int64_t* col_gids,
                   const double* vals, int is_complex, mxg_crs** out) {
  int layout = 0;
  if (const char* e = std::getenv("MXG_SPMV_LAYOUT")) layout = (std::strcmp(e, "sell") == 0) ? 1 : 0;
  return mxg_crs_create_opts(row_map, domain_map, rowptr, col_gids, vals, is_complex, layout, out);
}

int mxg_crs_destroy(mxg_crs* A) {
  if (!A) return MXG_OK;
  cudaSetDevice(A->ctx->device);
  cudaStreamSynchronize(A->ctx->stream);
  cudaStreamSynchronize(A->ctx->commStream);
  for (auto& g : A->graphs) cudaGraphExecDestroy(g.exec);
  for (void* o : A->p2p.opened) cudaIpcCloseMemHandle(o);
  if (A->p2p.ghost) cudaFree(A->p2p.ghost);
  if (A->p2p.flags) cudaFree(A->p2p.flags);
  if (A->p2p.done) cudaFree(A->p2p.done);
  if (A->p2p.trace) cudaFree(A->p2p.trace);
  if (A->p2p.dArgs) cudaFree(A->p2p.dArgs);
  void* ptrs[] = {A->dRowPat, A->dPatOff, A->dPat, A->dGenRow, A->dGenLen, A->dSlicePtr, A->dCol, A->dVal, A->dSendIdx, A->dSendBuf, A->dGhost, A->dInvDiag, A->dWinTiles};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  mxg_map_destroy(A->rowMap);
  mxg_map_destroy(A->domMap);
  delete A;
  return MXG_OK;
}

static int checkApply(const char* fn, const mxg_crs* A, const mxg_mv* x, const mxg_mv* y) {
  MXG_REQUIRE(A && x && y, "%s: NULL argument", fn);
  MXG_REQUIRE(x->map->ctx == A->ctx && y->map->ctx == A->ctx, "%s: operands live on different contexts", fn);
  MXG_REQUIRE(x->isComplex == A->isComplex && y->isComplex == A->isComplex, "%s: mixed real/complex operands", fn);
  MXG_REQUIRE(x->ld == A->nLoc, "%s: x has local length %lld, operator domain has %lld", fn, (long long)x->ld, (long long)A->nLoc);
  MXG_REQUIRE(y->ld == A->nRows, "%s: y has local length %lld, operator range has %lld", fn, (long long)y->ld, (long long)A->nRows);
  MXG_REQUIRE(x->ncols == y->ncols, "%s: x has %d columns, y has %d", fn, x->ncols, y->ncols);
  if (x->storage.get() == y->storage.get())
    for (void* px : x->col)
      for (void* py : y->col) MXG_REQUIRE(px != py, "%s: x and y must not alias", fn);
  return MXG_OK;
}

int mxg_crs_apply(const mxg_crs* A, const mxg_mv* x, mxg_mv* y) {
  int rc = checkApply("mxg_crs_apply", A, x, y);
  if (rc) return rc;
  MXG_CUDA(cudaSetDevice(A->ctx->device));
  if (A->isComplex) {
    Epilogue<zd> ep{{1, 0}, {0, 0}, 0};
    return applyImpl<zd>(A, x, y, ep);
  }
  Epilogue<double> ep{1.0, 0.0, 0};
  return applyImpl<double>(A, x, y, ep);
}

// Host-buffer batch apply: y_host[i] = A x_host[i]. Two device slots and two copy streams, so the upload of item
// i+1 and the download of item i-1 run while item i is applied (PCIe is full duplex); every item still crosses the
// bus in both directions. Returns when all results are in host memory.
int mxg_crs_apply_host_batch(const mxg_crs* A, int count, const double* const* x_host, double* const* y_host) {
  MXG_REQUIRE(A && (count == 0 || (x_host && y_host)), "mxg_crs_apply_host_batch: NULL argument");
  MXG_REQUIRE(count >= 0, "mxg_crs_apply_host_batch: negative count");
  if (count == 0) return MXG_OK;
  for (int i = 0; i < count; ++i) MXG_REQUIRE(x_host[i] && y_host[i], "mxg_crs_apply_host_batch: NULL buffer %d", i);
  mxg_ctx* ctx = A->ctx;
  MXG_REQUIRE(A->rowMap->perm.empty() && A->domMap->perm.empty(), "mxg_crs_apply_host_batch: operator lives on ordered maps");
  MXG_CUDA(cudaSetDevice(ctx->device));
  const size_t esz = A->isComplex ? 16 : 8;
  mxg_mv *xs[2] = {nullptr, nullptr}, *ys[2] = {nullptr, nullptr};
  cudaStream_t sUp = nullptr, sDown = nullptr;
  cudaEvent_t evUp[2] = {nullptr, nullptr}, evApply[2] = {nullptr, nullptr}, evDown[2] = {nullptr, nullptr};
  int rc = MXG_OK;
  cudaError_t e = cudaSuccess;
  auto ok = [&]() { return rc == MXG_OK && e == cudaSuccess; };
  for (int s = 0; s < 2 && ok(); ++s) {
    rc = mxg_mv_create(A->domMap, 1, A->isComplex, &xs[s]);
    if (rc == MXG_OK) rc = mxg_mv_create(A->rowMap, 1, A->isComplex, &ys[s]);
    if (ok()) e = cudaEventCreateWithFlags(&evUp[s], cudaEventDisableTiming);
    if (ok()) e = cudaEventCreateWithFlags(&evApply[s], cudaEventDisableTiming);
    if (ok()) e = cudaEventCreateWithFlags(&evDown[s], cudaEventDisableTiming);
  }
  if (ok()) e = cudaStreamCreateWithFlags(&sUp, cudaStreamNonBlocking);
  if (ok()) e = cudaStreamCreateWithFlags(&sDown, cudaStreamNonBlocking);
  for (int i = 0; i < count && ok(); ++i) {
    const int s = i & 1;
    // x slot is free once the apply of item i-2 has consumed it
    if (i >= 2) e = cudaStreamWaitEvent(sUp, evApply[s], 0);
    if (ok() && xs[s]->ld) e = cudaMemcpyAsync(xs[s]->col[0], x_host[i], size_t(xs[s]->ld) * esz, cudaMemcpyHostToDevice, sUp);
    if (ok()) e = cudaEventRecord(evUp[s], sUp);
    if (ok()) e = cudaStreamWaitEvent(ctx->stream, evUp[s], 0);
    // y slot is free once item i-2 has been downloaded
    if (ok() && i >= 2) e = cudaStreamWaitEvent(ctx->stream, evDown[s], 0);
    if (ok()) rc = mxg_crs_apply(A, xs[s], ys[s]);
    if (ok()) e = cudaEventRecord(evApply[s], ctx->stream);
    if (ok()) e = cudaStreamWaitEvent(sDown, evApply[s], 0);
    if (ok() && ys[s]->ld) e = cudaMemcpyAsync(y_host[i], ys[s]->col[0], size_t(ys[s]->ld) * esz, cudaMemcpyDeviceToHost, sDown);
    if (ok()) e = cudaEventRecord(evDown[s], sDown);
  }
  // drain everything before the slots are released, also on the error path
  if (sUp) cudaStreamSynchronize(sUp);
  cudaStreamSynchronize(ctx->stream);
  if (sDown) { cudaError_t e2 = cudaStreamSynchronize(sDown); if (e == cudaSuccess) e = e2; }
  for (int s = 0; s < 2; ++s) {
    if (evUp[s]) cudaEventDestroy(evUp[s]);
    if (evApply[s]) cudaEventDestroy(evApply[s]);
    if (evDown[s]) cudaEventDestroy(evDown[s]);
    if (xs[s]) mxg_mv_destroy(xs[s]);
    if (ys[s]) mxg_mv_destroy(ys[s]);
  }
  if (sUp) cudaStreamDestroy(sUp);
  if (sDown) cudaStreamDestroy(sDown);
  if (rc != MXG_OK) return rc;
  MXG_REQUIRE(e == cudaSuccess, "mxg_crs_apply_host_batch: %s", cudaGetErrorString(e));
  return MXG_OK;
}

int mxg_crs_apply_axpby(const mxg_crs* A, const double alpha[2], const mxg_mv* x, const double beta[2], mxg_mv* y) {
  int rc = checkApply("mxg_crs_apply_axpby", A, x, y);
  if (rc) return rc;
  MXG_REQUIRE(alpha && beta, "mxg_crs_apply_axpby: NULL scalar");
  MXG_CUDA(cudaSetDevice(A->ctx->device));
  if (A->isComplex) {
    Epilogue<zd> ep{scalarOf<zd>(alpha), scalarOf<zd>(beta), 1};
    return applyImpl<zd>(A, x, y, ep);
  }
  Epilogue<double> ep{alpha[0], beta[0], 1};
  return applyImpl<double>(A, x, y, ep);
}

int mxg_crs_apply_timed(const mxg_crs* A, const mxg_mv* x, mxg_mv* y, double ms[4]) {
  MXG_REQUIRE(ms, "mxg_crs_apply_timed: NULL argument");
  int rc = checkApply("mxg_crs_apply_timed", A, x, y);
  if (rc) return rc;
  mxg_ctx* ctx = A->ctx;
  MXG_CUDA(cudaSetDevice(ctx->device));
  for (auto& e : ctx->prof)
    if (!e) MXG_CUDA(cudaEventCreate(&e));
  // the single launch is one kernel: its phases come from the %globaltimer marks of its roles, not from events
  const bool peer = peerLaunch(A, x->ncols);
  if (peer) {
    rc = mxg_crs_trace(A, 1, nullptr);
    if (rc) return rc;
  }
  auto timedApply = [&]() -> int {
    MXG_CUDA(cudaEventRecord(ctx->prof[0], ctx->stream));
    ctx->profiling = true;
    const int rcApply = mxg_crs_apply(A, x, y);
    ctx->profiling = false;
    if (rcApply) return rcApply;
    MXG_CUDA(cudaEventRecord(ctx->prof[4], ctx->stream));
    MXG_CUDA(cudaEventSynchronize(ctx->prof[4]));
    MXG_CUDA(cudaStreamSynchronize(ctx->commStream));
    return MXG_OK;
  };
  rc = timedApply();
  double t[10];
  if (peer) {   // read back and disarm, also when the apply failed
    const int rcTrace = mxg_crs_trace(A, 0, t);
    if (!rc) rc = rcTrace;
  }
  if (rc) return rc;
  float f = 0;
  ms[0] = ms[1] = ms[2] = 0;
  const bool halo = ctx->nranks > 1 && (A->gLo + A->gHi > 0 || A->sendTotal > 0);
  if (peer) {
    // first start to last end over roles r0..r1, ns -> ms; a role that did not run (-1) counts 0
    auto span = [&t](int r0, int r1) {
      double lo = -1, hi = -1;
      for (int r = r0; r <= r1; ++r) {
        if (t[2 * r] < 0) continue;
        if (lo < 0 || t[2 * r] < lo) lo = t[2 * r];
        if (t[2 * r + 1] > hi) hi = t[2 * r + 1];
      }
      return lo < 0 ? 0.0 : (hi - lo) * 1e-6;
    };
    ms[0] = span(1, 2);   // interior dictionary + sliced-ELL rows
    ms[1] = span(4, 4);   // boundary rows
    ms[2] = span(0, 0);   // pack + flag publish
  } else if (!halo) {
    MXG_CUDA(cudaEventElapsedTime(&f, ctx->prof[1], ctx->prof[2])); ms[0] = f;   // dictionary kernel
    MXG_CUDA(cudaEventElapsedTime(&f, ctx->prof[2], ctx->prof[3])); ms[1] = f;   // sliced-ELL kernel
    MXG_CUDA(cudaEventElapsedTime(&f, ctx->prof[0], ctx->prof[1])); ms[2] = f;
  } else {
    MXG_CUDA(cudaEventElapsedTime(&f, ctx->prof[5], ctx->prof[4])); ms[0] = f;   // interior rows (+ final wait)
    MXG_CUDA(cudaEventElapsedTime(&f, ctx->prof[2], ctx->prof[3])); ms[1] = f;   // boundary rows
    MXG_CUDA(cudaEventElapsedTime(&f, ctx->prof[1], ctx->prof[2])); ms[2] = f;   // NCCL send/recv
  }
  MXG_CUDA(cudaEventElapsedTime(&f, ctx->prof[0], ctx->prof[4])); ms[3] = f;
  return MXG_OK;
}

// %globaltimer timeline of the fused multi-rank apply. enable != 0: arm (allocate / reset) the trace buffer; enable == 0:
// read it back into out[10] (ns relative to the earliest mark; role r: out[2r] = first start, out[2r+1] = last end; roles:
// 0 pack + publish, 1 interior dictionary rows, 2 interior sliced-ELL rows, 3 boundary blocks waiting for the neighbours'
// flags, 4 boundary rows) and disarm.
int mxg_crs_trace(const mxg_crs* A, int enable, double out[10]) {
  MXG_REQUIRE(A, "mxg_crs_trace: NULL argument");
  mxg_ctx* ctx = A->ctx;
  MXG_CUDA(cudaSetDevice(ctx->device));
  auto& q = A->p2p;
  unsigned long long init[10];
  for (int r = 0; r < 5; ++r) { init[2 * r] = ~0ull; init[2 * r + 1] = 0ull; }
  if (enable) {
    if (!q.trace) MXG_CUDA(cudaMalloc(&q.trace, sizeof(init)));
    MXG_CUDA(cudaMemcpyAsync(q.trace, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
    MXG_CUDA(cudaStreamSynchronize(ctx->stream));
    return MXG_OK;
  }
  MXG_REQUIRE(q.trace && out, "mxg_crs_trace: trace not armed");
  unsigned long long h[10];
  MXG_CUDA(cudaStreamSynchronize(ctx->stream));
  MXG_CUDA(cudaMemcpy(h, q.trace, sizeof(h), cudaMemcpyDeviceToHost));
  unsigned long long t0 = ~0ull;
  for (int r = 0; r < 5; ++r) if (h[2 * r] < t0) t0 = h[2 * r];
  for (int r = 0; r < 5; ++r) {
    out[2 * r] = h[2 * r] == ~0ull ? -1.0 : double(h[2 * r] - t0);
    out[2 * r + 1] = h[2 * r + 1] == 0ull ? -1.0 : double(h[2 * r + 1] - t0);
  }
  MXG_CUDA(cudaFree(q.trace));
  q.trace = nullptr;
  return MXG_OK;
}

int mxg_crs_stats(const mxg_crs* A, int64_t out[8]) {
  MXG_REQUIRE(A && out, "mxg_crs_stats: NULL argument");
  out[0] = A->nRows;
  out[1] = A->nnz;
  out[2] = A->dictRows;
  out[3] = A->numPats;
  out[4] = int64_t(A->deviceBytes);
  out[5] = A->gLo + A->gHi;
  out[6] = A->ghostRows;
  out[7] = A->ellEntries;
  return MXG_OK;
}

}  // extern "C"
