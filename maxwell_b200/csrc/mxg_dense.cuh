// Tall-skinny dense block products of the eigensolver (real FP64): the Gram product C = A^T X (MvTransMv,
// src/MxAnasaziMV.cpp:114-149) and the update Y = alpha A B + beta Y (MvTimesMatAddMv, :8-33).
//
// Both kernels stream A (and X) exactly once through shared memory: the rows are cut into chunks of kDenseRows, one 1-D TMA
// copy (cp.async.bulk) per column segment fills a stage, two stages alternate behind mbarriers, and each CTA walks the
// chunks ch = blockIdx, blockIdx + gridDim, ... The contraction runs on the FP64 tensor path (mma.sync.m8n8k4.f64, DMMA):
// tcgen05 has no FP64 kind, and one 8-byte shared load per lane feeds 8 FMAs per lane, where the FMA-pipe kernels of
// round 2 sat at 95 % of the shared-memory wavefront limit and were 1.3-2.0x slower on every timed shape
// (profiles/README_r02.md section 2). The complex products and updates with more than kUpdateMaxK source columns run on the
// register-tiled kernels of mxg_mvops.cu.
#pragma once
#include "mxg_internal.h"
#include "mxg_spmm_win.cuh"

namespace mxg {

constexpr int kDenseRows = 64;                 // rows per pipeline stage
constexpr int kDenseStride = kDenseRows + 4;   // shared column stride (doubles): 544 B = 32 mod 128 -> the 4 columns x 4 rows a half
                                               // warp reads per DMMA fragment land in 16 distinct 8-byte bank pairs
constexpr int kDenseThreads = 256;

#ifdef __CUDACC__
// column segment [r0, r0 + rows) of `col` -> shared; every issuing thread arrives on the stage barrier with its own byte count
__device__ __forceinline__ void denseIssue(const double* col, int64_t r0, int rows, double* dst, uint64_t* bar) {
  const uint32_t bytes = uint32_t((rows * 8 + 15) & ~15);   // allocations are padded to 256 B: the extra element is in bounds
  mbarExpectTx(bar, bytes);
  bulkLoad(dst, col + r0, bytes, bar);
}

// ---- FP64 tensor-core contraction (mma.sync.m8n8k4.f64) --------------------------------------------------------------------
// Fragment layout (PTX ISA, m8n8k4): a0 = A[g][t], b0 = B[t][g], c0/c1 = C[g][2t], C[g][2t+1] with g = lane / 4, t = lane % 4.
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// Gram, C tile (16 RI) x (16 RJ): warp (wk, wm, wn) takes rows [32 wk, 32 wk + 32) of the chunk and the fragments
// [RI wm, RI wm + RI) x [RJ wn, RJ wn + RJ); the two row halves are written as separate partial slices.
template <int RI, int RJ>
__global__ void __launch_bounds__(kDenseThreads, 2) k_gram_mma(ColTable<double> A, int k, ColTable<double> X, int b, int64_t n, int tilesB,
                                                               double* __restrict__ partial) {
  constexpr int TI = 16 * RI, TJ = 16 * RJ, NC = TI + TJ;
  extern __shared__ __align__(128) unsigned char smemRaw[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smemRaw);
  double* stage0 = reinterpret_cast<double*>(smemRaw + 128);
  constexpr int stageElems = NC * kDenseStride;
  const int tk = blockIdx.x / tilesB, tb = blockIdx.x % tilesB;
  const int k0 = tk * TI, b0 = tb * TJ;
  const int kc = min(TI, k - k0), bc = min(TJ, b - b0);
  const int nIssue = kc + bc;
  const int t = threadIdx.x;
  if (t == 0) {
    mbarInit(&bar[0], nIssue);
    mbarInit(&bar[1], nIssue);
    mbarFenceInit();
  }
  __syncthreads();
  const int64_t chunks = (n + kDenseRows - 1) / kDenseRows;
  const double* myCol = nullptr;
  int mySlot = 0;
  if (t < kc) { myCol = A.p[k0 + t]; mySlot = t; }
  else if (t < nIssue) { myCol = X.p[b0 + (t - kc)]; mySlot = TI + (t - kc); }
  auto issue = [&](int64_t ch, int s) {
    if (myCol) {
      const int64_t r0 = ch * kDenseRows;
      const int rows = int(min(int64_t(kDenseRows), n - r0));
      denseIssue(myCol, r0, rows, stage0 + s * stageElems + mySlot * kDenseStride, &bar[s]);
    }
  };
  const int warp = t >> 5, lane = t & 31;
  const int g = lane >> 2, tg = lane & 3;
  const int wk = warp >> 2, wm = (warp >> 1) & 1, wn = warp & 1;
  double acc[RI][RJ][2];
#pragma unroll
  for (int i = 0; i < RI; ++i)
#pragma unroll
    for (int j = 0; j < RJ; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  int64_t ch = blockIdx.y;
  if (ch < chunks) issue(ch, 0);
  int it = 0;
  for (; ch < chunks; ch += gridDim.y, ++it) {
    const int s = it & 1;
    const int64_t next = ch + gridDim.y;
    if (next < chunks) issue(next, s ^ 1);
    mbarWait(&bar[s], (it >> 1) & 1);
    double* sA = stage0 + s * stageElems;
    const int64_t r0 = ch * kDenseRows;
    if (n - r0 < kDenseRows) {                              // tail chunk: rows past the end contribute zero
      const int valid = int(n - r0);
      for (int e = t; e < NC * kDenseRows; e += kDenseThreads) {
        const int c = e / kDenseRows, r = e % kDenseRows;
        if (r >= valid) sA[c * kDenseStride + r] = 0.0;
      }
      __syncthreads();
    }
    const double* pa = sA + (8 * RI * wm + g) * kDenseStride + 32 * wk + tg;
    const double* px = sA + (TI + 8 * RJ * wn + g) * kDenseStride + 32 * wk + tg;
#pragma unroll
    for (int r = 0; r < 32; r += 4) {
      double av[RI], xv[RJ];
#pragma unroll
      for (int i = 0; i < RI; ++i) av[i] = pa[8 * i * kDenseStride + r];
#pragma unroll
      for (int j = 0; j < RJ; ++j) xv[j] = px[8 * j * kDenseStride + r];
#pragma unroll
      for (int i = 0; i < RI; ++i)
#pragma unroll
        for (int j = 0; j < RJ; ++j) dmma884(acc[i][j][0], acc[i][j][1], av[i], xv[j]);
    }
    __syncthreads();
  }
  const int slices = 2 * gridDim.y, slice = 2 * blockIdx.y + wk;
#pragma unroll
  for (int i = 0; i < RI; ++i)
#pragma unroll
    for (int j = 0; j < RJ; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int ci = 8 * (RI * wm + i) + g, cj = 8 * (RJ * wn + j) + 2 * tg + e;
        if (ci < kc && cj < bc) partial[(int64_t(k0 + ci) + int64_t(b0 + cj) * k) * slices + slice] = acc[i][j][e];
      }
}

// update: chunk of 64 rows = 8 row fragments; warp (wr, wc) takes row fragments 2 wr, 2 wr + 1 and the column fragments
// [RC wc, RC wc + RC). k is padded to a multiple of 4 with zero coefficient rows (and zeroed A slots).
template <int RC>
__global__ void __launch_bounds__(kDenseThreads, 2) k_update_mma(ColTable<double> A, int k, const double* __restrict__ Bg, int b, double alpha,
                                                                 double beta, ColTable<double> Y, int64_t n) {
  extern __shared__ __align__(128) unsigned char smemRaw[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smemRaw);
  double* sB = reinterpret_cast<double*>(smemRaw + 128);        // [k4][BW]
  constexpr int BW = 16 * RC + 4;                                // 20 / 36 / 52 doubles: 32 mod 128 bytes -> conflict-free fragments
  const int k4 = (k + 3) & ~3;
  double* stage0 = sB + ((k4 * BW + 15) & ~15);
  const int stageElems = k4 * kDenseStride;
  const int t = threadIdx.x;
  if (t == 0) {
    mbarInit(&bar[0], k);
    mbarInit(&bar[1], k);
    mbarFenceInit();
  }
  for (int e = t; e < k4 * BW; e += kDenseThreads) {
    const int i = e / BW, j = e % BW;
    sB[e] = (i < k && j < b) ? Bg[i + int64_t(j) * k] : 0.0;
  }
  for (int e = t; e < 2 * (k4 - k) * kDenseStride; e += kDenseThreads) {    // padded A columns: 0 * garbage could be NaN
    const int s = e / ((k4 - k) * kDenseStride), r = e % ((k4 - k) * kDenseStride);
    stage0[s * stageElems + k * kDenseStride + r] = 0.0;
  }
  __syncthreads();
  const int64_t chunks = (n + kDenseRows - 1) / kDenseRows;
  auto issue = [&](int64_t ch, int s) {
    for (int c = t; c < k; c += kDenseThreads) {
      const int64_t r0 = ch * kDenseRows;
      const int rows = int(min(int64_t(kDenseRows), n - r0));
      denseIssue(A.p[c], r0, rows, stage0 + s * stageElems + c * kDenseStride, &bar[s]);
    }
  };
  const int warp = t >> 5, lane = t & 31;
  const int g = lane >> 2, tg = lane & 3;
  const int wr = warp >> 1, wc = warp & 1;
  int64_t ch = blockIdx.x;
  if (ch < chunks) issue(ch, 0);
  int it = 0;
  for (; ch < chunks; ch += gridDim.x, ++it) {
    const int s = it & 1;
    const int64_t next = ch + gridDim.x;
    if (next < chunks) issue(next, s ^ 1);
    mbarWait(&bar[s], (it >> 1) & 1);
    const double* pa = stage0 + s * stageElems + tg * kDenseStride + 16 * wr + g;
    const double* pb = sB + tg * BW + 8 * RC * wc + g;
    double acc[2][RC][2];
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
      for (int j = 0; j < RC; ++j) acc[m][j][0] = acc[m][j][1] = 0.0;
#pragma unroll 2
    for (int i = 0; i < k4; i += 4) {
      const double a0 = pa[i * kDenseStride], a1 = pa[i * kDenseStride + 8];
      double bv[RC];
#pragma unroll
      for (int j = 0; j < RC; ++j) bv[j] = pb[i * BW + 8 * j];
#pragma unroll
      for (int j = 0; j < RC; ++j) {
        dmma884(acc[0][j][0], acc[0][j][1], a0, bv[j]);
        dmma884(acc[1][j][0], acc[1][j][1], a1, bv[j]);
      }
    }
    const int64_t rbase = ch * kDenseRows + 16 * wr + g;
#pragma unroll
    for (int j = 0; j < RC; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int c = 8 * (RC * wc + j) + 2 * tg + e;
        if (c < b) {
          double* y = Y.p[c];
#pragma unroll
          for (int m = 0; m < 2; ++m) {
            const int64_t row = rbase + 8 * m;
            if (row < n) {
              double v = alpha * acc[m][j][e];
              if (beta != 0.0) v += beta * y[row];
              y[row] = v;
            }
          }
        }
      }
    __syncthreads();
  }
}
#endif

}  // namespace mxg
