// libmxgpu: multivector block operations (K5-K14 of SURVEY.md section 2.3). All kernels are
// HBM-bound streaming or reduction kernels; grids are sized in multiples of the SM count.
#include <cmath>
#include <cstring>

#include "mxg_internal.h"
#include "mxg_dense.cuh"

using namespace mxg;

namespace {

constexpr int kBlock = 256;

template <class T>
struct ScalarList {
  T v[MXG_MAX_COLS];
};

// ---- elementwise -------------------------------------------------------------------------
template <class T>
__global__ void __launch_bounds__(kBlock) k_fill(ColTable<T> t, int64_t n, T alpha) {
  T* __restrict__ c = t.p[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock) c[i] = alpha;
}

template <class T>
__global__ void __launch_bounds__(kBlock) k_scale_cols(ColTable<T> t, int64_t n, ScalarList<T> a) {
  T* __restrict__ c = t.p[blockIdx.y];
  const T s = a.v[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock) c[i] = s * c[i];
}

__global__ void __launch_bounds__(kBlock) k_conj(ColTable<zd> t, int64_t n) {
  zd* __restrict__ c = t.p[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock) c[i].y = -c[i].y;
}

// dst = a*A + b*B. Pure elementwise, so A or B may alias dst. A zero coefficient drops its
// operand entirely (Epetra_MultiVector::Update semantics).
template <class T, bool USE_A, bool USE_B>
__global__ void __launch_bounds__(kBlock) k_axpby(ColTable<T> d, T a, ColTable<T> A, T b, ColTable<T> B, int64_t n) {
  T* dst = d.p[blockIdx.y];
  const T* pa = A.p[blockIdx.y];
  const T* pb = B.p[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock) {
    T r = zeroOf<T>();
    if (USE_A) r = a * pa[i];
    if (USE_B) { T tb = b * pb[i]; r = USE_A ? r + tb : tb; }
    dst[i] = r;
  }
}

template <class T>
__global__ void __launch_bounds__(kBlock) k_copy(ColTable<T> d, ColTable<T> s, int64_t n) {
  T* __restrict__ dst = d.p[blockIdx.y];
  const T* __restrict__ src = s.p[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock) dst[i] = src[i];
}

// Counter-based generator: uniform (-1,1) from a hash of (seed, global DOF id, column, re/im).
__host__ __device__ inline double hashUniform(uint64_t seed, uint64_t gid, uint64_t col, uint64_t part) {
  uint64_t z = seed ^ (gid * 0x9E3779B97F4A7C15ull) ^ ((col + 1) * 0xBF58476D1CE4E5B9ull) ^ (part * 0x94D049BB133111EBull);
  z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
  z ^= z >> 27; z *= 0x94D049BB133111EBull;
  z ^= z >> 31;
  return 2.0 * (double(z >> 11) * (1.0 / 9007199254740992.0)) - 1.0;
}
struct ColIds {
  int v[MXG_MAX_COLS];
};
__global__ void __launch_bounds__(kBlock) k_random_real(ColTable<double> t, ColIds ids, const int64_t* __restrict__ gids, int64_t n, uint64_t seed) {
  double* __restrict__ c = t.p[blockIdx.y];
  const uint64_t col = ids.v[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock)
    c[i] = hashUniform(seed, uint64_t(gids[i]), col, 0);
}
__global__ void __launch_bounds__(kBlock) k_random_cplx(ColTable<zd> t, ColIds ids, const int64_t* __restrict__ gids, int64_t n, uint64_t seed) {
  zd* __restrict__ c = t.p[blockIdx.y];
  const uint64_t col = ids.v[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock)
    c[i] = {hashUniform(seed, uint64_t(gids[i]), col, 0), hashUniform(seed, uint64_t(gids[i]), col, 1)};
}

// ---- reductions --------------------------------------------------------------------------
__device__ inline double warpSum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ inline zd warpSum(zd v) { return {warpSum(v.x), warpSum(v.y)}; }

template <class T>
__device__ inline T blockSum(T v, T* sm /* kBlock/32 entries */) {
  v = warpSum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sm[w] = v;
  __syncthreads();
  T r = zeroOf<T>();
  if (w == 0) {
    r = l < kBlock / 32 ? sm[l] : zeroOf<T>();
    r = warpSum(r);
  }
  return r;  // valid in warp 0
}

// partial[col * gridDim.x + block] = sum over this block's rows of conj(a) * b
template <class T>
__global__ void __launch_bounds__(kBlock) k_dot_partial(ColTable<T> A, ColTable<T> B, int64_t n, T* __restrict__ partial) {
  __shared__ T sm[kBlock / 32];
  const T* __restrict__ a = A.p[blockIdx.y];
  const T* __restrict__ b = B.p[blockIdx.y];
  T acc0 = zeroOf<T>(), acc1 = zeroOf<T>();
  const int64_t stride = int64_t(gridDim.x) * kBlock;
  int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x;
  for (; i + stride < n; i += 2 * stride) {
    fmaInto(acc0, conjz(a[i]), b[i]);
    fmaInto(acc1, conjz(a[i + stride]), b[i + stride]);
  }
  if (i < n) fmaInto(acc0, conjz(a[i]), b[i]);
  T r = blockSum(acc0 + acc1, sm);
  if (threadIdx.x == 0) partial[blockIdx.y * int64_t(gridDim.x) + blockIdx.x] = r;
}

// out[item] = sum_{p < np} partial[item * np + p], fixed order -> deterministic
template <class T>
__global__ void __launch_bounds__(kBlock) k_reduce_partials(const T* __restrict__ partial, int np, T* __restrict__ out) {
  __shared__ T sm[kBlock / 32];
  T acc = zeroOf<T>();
  for (int p = threadIdx.x; p < np; p += kBlock) acc += partial[blockIdx.x * int64_t(np) + p];
  T r = blockSum(acc, sm);
  if (threadIdx.x == 0) out[blockIdx.x] = r;
}

// dst_j = a_j * A_j + b_j * B_j with one scalar pair per column (the CG / Chebyshev recurrences: x += alpha_j p,
// r -= alpha_j q, p = z + beta_j p in ONE kernel each instead of copy + MvScale(vector) + MvAddMv). A or B may alias dst.
template <class T>
__global__ void __launch_bounds__(kBlock) k_axpby_cols(ColTable<T> d, ScalarList<T> a, ColTable<T> A, ScalarList<T> b, ColTable<T> B, int64_t n) {
  T* dst = d.p[blockIdx.y];
  const T* pa = A.p[blockIdx.y];
  const T* pb = B.p[blockIdx.y];
  const T sa = a.v[blockIdx.y], sb = b.v[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock) dst[i] = sa * pa[i] + sb * pb[i];
}

// partial[col * gridDim.x + block] = sum over this block's rows of a
template <class T>
__global__ void __launch_bounds__(kBlock) k_sum_partial(ColTable<T> A, int64_t n, T* __restrict__ partial) {
  __shared__ T sm[kBlock / 32];
  const T* __restrict__ a = A.p[blockIdx.y];
  T acc = zeroOf<T>();
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock) acc += a[i];
  T r = blockSum(acc, sm);
  if (threadIdx.x == 0) partial[blockIdx.y * int64_t(gridDim.x) + blockIdx.x] = r;
}
// x_j -= sums[j] / count (sums stay on the device: no host round trip between the reduction and the update)
template <class T>
__global__ void __launch_bounds__(kBlock) k_sub_mean(ColTable<T> X, const T* __restrict__ sums, double invCount, int64_t n) {
  T* __restrict__ x = X.p[blockIdx.y];
  const T s = sums[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock) {
    T v = x[i];
    if constexpr (sizeof(T) == sizeof(double)) v = v - s * invCount;
    else { v.x -= s.x * invCount; v.y -= s.y * invCount; }
    x[i] = v;
  }
}
// x_j[i] = 0 where frac[i] == 0 (MxGridField::zeroUnusedComponents)
template <class T>
__global__ void __launch_bounds__(kBlock) k_zero_unused(ColTable<T> X, const double* __restrict__ frac, int fracStride, int64_t n) {
  T* __restrict__ x = X.p[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock)
    if (frac[i * fracStride] == 0.0) x[i] = zeroOf<T>();
}

// ---- tall-skinny Gram product: C(k x b) = A^H X ---------------------------------------------
// Each thread owns a KT x BT register tile of C and streams rows with stride kBlock (coalesced
// per column). blockIdx.x enumerates tiles (fastest), blockIdx.y row slices: blocks that share
// rows are co-scheduled so the re-read of A/X columns by other tiles is served from L2.
template <class T, int KT, int BT>
__global__ void __launch_bounds__(kBlock) k_trans_mv(ColTable<T> A, int k, ColTable<T> X, int b, int64_t n,
                                                     int tilesB, T* __restrict__ partial /* [gridDim.y][k*b] */) {
  __shared__ T sm[kBlock / 32];
  const int tk = blockIdx.x / tilesB, tb = blockIdx.x % tilesB;
  const int k0 = tk * KT, b0 = tb * BT;
  const T* pa[KT];
  const T* px[BT];
#pragma unroll
  for (int i = 0; i < KT; ++i) pa[i] = A.p[min(k0 + i, k - 1)];
#pragma unroll
  for (int j = 0; j < BT; ++j) px[j] = X.p[min(b0 + j, b - 1)];
  T acc[KT][BT];
#pragma unroll
  for (int i = 0; i < KT; ++i)
#pragma unroll
    for (int j = 0; j < BT; ++j) acc[i][j] = zeroOf<T>();
  for (int64_t r = blockIdx.y * int64_t(kBlock) + threadIdx.x; r < n; r += int64_t(gridDim.y) * kBlock) {
    T av[KT], xv[BT];
#pragma unroll
    for (int i = 0; i < KT; ++i) av[i] = conjz(pa[i][r]);
#pragma unroll
    for (int j = 0; j < BT; ++j) xv[j] = px[j][r];
#pragma unroll
    for (int i = 0; i < KT; ++i)
#pragma unroll
      for (int j = 0; j < BT; ++j) fmaInto(acc[i][j], av[i], xv[j]);
  }
#pragma unroll
  for (int i = 0; i < KT; ++i)
#pragma unroll
    for (int j = 0; j < BT; ++j) {
      T r = blockSum(acc[i][j], sm);
      if (threadIdx.x == 0 && k0 + i < k && b0 + j < b)
        partial[(int64_t(k0 + i) + int64_t(b0 + j) * k) * gridDim.y + blockIdx.y] = r;
    }
}

// ---- tall-skinny update: Y = alpha * A * B + beta * Y ---------------------------------------
// The small dense B rides in the kernel parameter block (constant bank): the FMAs take it as a
// uniform operand, so the only memory instructions are the streaming loads of A and Y.
constexpr int kUpdateMaxK = 64;   // widest A the TMA-staged update kernel takes (shared memory: 2 stages of k columns + B)
constexpr int kMaxBParam = 1536;  // doubles (12 KB of the 32 KB parameter space)
struct DenseParam {
  double v[kMaxBParam];
};
__device__ inline double denseAt(const DenseParam& B, int idx, double) { return B.v[idx]; }
__device__ inline zd denseAt(const DenseParam& B, int idx, zd) { return {B.v[2 * idx], B.v[2 * idx + 1]}; }

// B (k x bcount) is copied from the parameter block into shared memory as [i][j] (j fastest), so
// the inner loop reads it with warp-wide broadcast loads; every thread owns RT rows x BT columns of
// the result in registers (one B value feeds RT FMAs, one A value feeds BT FMAs).
template <class T, int BT, int RT>
__global__ void __launch_bounds__(kBlock) k_times_mat(ColTable<T> A, int k, const __grid_constant__ DenseParam B, int b0, int bcount,
                                                      T alpha, T beta, bool useY, ColTable<T> Y, int64_t n) {
  extern __shared__ __align__(16) unsigned char smemRaw[];
  T* sB = reinterpret_cast<T*>(smemRaw);   // [k][BT]
  for (int t = threadIdx.x; t < k * BT; t += kBlock) {
    const int i = t / BT, j = t % BT;
    sB[t] = j < bcount ? denseAt(B, i + (b0 + j) * k, T()) : zeroOf<T>();
  }
  __syncthreads();
  const int64_t tile = int64_t(kBlock) * RT;
  for (int64_t base = blockIdx.x * tile; base < n; base += int64_t(gridDim.x) * tile) {
    int64_t r[RT];
    bool ok[RT];
#pragma unroll
    for (int t = 0; t < RT; ++t) { r[t] = base + t * kBlock + threadIdx.x; ok[t] = r[t] < n; if (!ok[t]) r[t] = n - 1; }
    T acc[RT][BT];
#pragma unroll
    for (int t = 0; t < RT; ++t)
#pragma unroll
      for (int j = 0; j < BT; ++j) acc[t][j] = zeroOf<T>();
#pragma unroll 2
    for (int i = 0; i < k; ++i) {
      T a[RT];
      const T* col = A.p[i];
#pragma unroll
      for (int t = 0; t < RT; ++t) a[t] = col[r[t]];
#pragma unroll
      for (int j = 0; j < BT; ++j) {
        const T bv = sB[i * BT + j];
#pragma unroll
        for (int t = 0; t < RT; ++t) fmaInto(acc[t][j], a[t], bv);
      }
    }
#pragma unroll
    for (int j = 0; j < BT; ++j)
      if (j < bcount) {
        T* y = Y.p[b0 + j];
#pragma unroll
        for (int t = 0; t < RT; ++t)
          if (ok[t]) {
            T v = alpha * acc[t][j];
            if (useY) v = v + beta * y[r[t]];
            y[r[t]] = v;
          }
      }
  }
}

template <class T>
dim3 gridCols(const mxg_ctx* ctx, int64_t n, int ncols) {
  int perCol = gridFor(ctx, n, kBlock * 4, 8);
  int cap = (ctx->numSMs * 8 + ncols - 1) / ncols;
  if (perCol > cap) perCol = cap;
  if (perCol < 1) perCol = 1;
  return dim3(perCol, ncols);
}

#define LAUNCH_CHECK(ctx)                   \
  do {                                      \
    (ctx)->launches++;                      \
    MXG_CUDA(cudaGetLastError());           \
  } while (0)

template <class T>
int fillImpl(mxg_mv* mv, const double alpha[2]) {
  mxg_ctx* ctx = mv->map->ctx;
  if (mv->ld == 0) return MXG_OK;
  k_fill<T><<<gridCols<T>(ctx, mv->ld, mv->ncols), kBlock, 0, ctx->stream>>>(tableOf<T>(mv), mv->ld, scalarOf<T>(alpha));
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}

template <class T>
int scaleColsImpl(mxg_mv* mv, const double* alphas, bool same) {
  mxg_ctx* ctx = mv->map->ctx;
  if (mv->ld == 0) return MXG_OK;
  ScalarList<T> a;
  constexpr int w = sizeof(T) / sizeof(double);
  for (int j = 0; j < mv->ncols; ++j) {
    double s[2] = {alphas[same ? 0 : j * w], w == 2 ? alphas[same ? 1 : j * w + 1] : 0.0};
    a.v[j] = scalarOf<T>(s);
  }
  k_scale_cols<T><<<gridCols<T>(ctx, mv->ld, mv->ncols), kBlock, 0, ctx->stream>>>(tableOf<T>(mv), mv->ld, a);
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}

template <class T>
int axpbyImpl(mxg_mv* dst, const double alpha[2], const mxg_mv* A, const double beta[2], const mxg_mv* B) {
  mxg_ctx* ctx = dst->map->ctx;
  if (dst->ld == 0) return MXG_OK;
  const T a = scalarOf<T>(alpha), b = scalarOf<T>(beta);
  const bool ua = !isZero(a), ub = !isZero(b);
  const dim3 grid = gridCols<T>(ctx, dst->ld, dst->ncols);
  auto d = tableOf<T>(dst), ta = tableOf<T>(A), tb = tableOf<T>(B);
  if (ua && ub) k_axpby<T, true, true><<<grid, kBlock, 0, ctx->stream>>>(d, a, ta, b, tb, dst->ld);
  else if (ua) k_axpby<T, true, false><<<grid, kBlock, 0, ctx->stream>>>(d, a, ta, b, tb, dst->ld);
  else if (ub) k_axpby<T, false, true><<<grid, kBlock, 0, ctx->stream>>>(d, a, ta, b, tb, dst->ld);
  else k_axpby<T, false, false><<<grid, kBlock, 0, ctx->stream>>>(d, a, ta, b, tb, dst->ld);
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}

// column-wise conj(a_j).b_j into ctx->dScratch[0 .. ncols*w), all-reduced; leaves the result on the device
template <class T>
int dotToScratch(const mxg_mv* a, const mxg_mv* b) {
  mxg_ctx* ctx = a->map->ctx;
  const int nc = a->ncols;
  constexpr int w = sizeof(T) / sizeof(double);
  int np = gridFor(ctx, a->ld, kBlock * 8, 4);
  int cap = (ctx->numSMs * 4 + nc - 1) / nc;
  if (np > cap) np = cap;
  if (np < 1) np = 1;
  int rc = ensureScratch(ctx, sizeof(T) * (size_t(nc) * np + nc));
  if (rc) return rc;
  T* out = reinterpret_cast<T*>(ctx->dScratch);
  T* partial = out + nc;
  k_dot_partial<T><<<dim3(np, nc), kBlock, 0, ctx->stream>>>(tableOf<T>(a), tableOf<T>(b), a->ld, partial);
  LAUNCH_CHECK(ctx);
  k_reduce_partials<T><<<nc, kBlock, 0, ctx->stream>>>(partial, np, out);
  LAUNCH_CHECK(ctx);
  return allReduceScratch(ctx, size_t(nc) * w);
}

int fetchScratch(mxg_ctx* ctx, double* host, size_t count) {
  int rc = ensurePinned(ctx, count * sizeof(double));
  if (rc) return rc;
  MXG_CUDA(cudaMemcpyAsync(ctx->hPinned, ctx->dScratch, count * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  {
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    rc = checkHaloFault(ctx, "reduction");
    if (rc) return rc;
    MXG_CUDA(e);
  }
  std::memcpy(host, ctx->hPinned, count * sizeof(double));
  return MXG_OK;
}

template <class T>
int transMvImpl(const double alpha[2], const mxg_mv* A, const mxg_mv* X, double* B, int ldb) {
  mxg_ctx* ctx = A->map->ctx;
  constexpr int w = sizeof(T) / sizeof(double);
  constexpr int KT = (w == 1) ? 8 : 4, BT = 4;
  const int k = A->ncols, b = X->ncols;
  const int tilesK = (k + KT - 1) / KT, tilesB = (b + BT - 1) / BT;
  const int tiles = tilesK * tilesB;
  int slices = (ctx->numSMs * 4 + tiles - 1) / tiles;
  int maxSlices = int((A->ld + kBlock - 1) / kBlock);
  if (slices > maxSlices) slices = maxSlices;
  if (slices < 1) slices = 1;
  const size_t kb = size_t(k) * b;
  // TMA-staged DMMA kernel (real case): the block tile of C is (16 ri) x (16 rj) with ri, rj in 1..3, chosen to cover k and b
  // with as little padding as possible
  const int ri = k >= 33 ? 3 : (k + 15) / 16, rj = b >= 33 ? 3 : (b + 15) / 16;   // block tile (16 ri) x (16 rj), at most 48 x 48
  const int gtB = (b + 16 * rj - 1) / (16 * rj), gtiles = ((k + 16 * ri - 1) / (16 * ri)) * gtB;
  int gs = (ctx->numSMs * 2 + gtiles - 1) / gtiles;
  {
    const int64_t chunks = (A->ld + kDenseRows - 1) / kDenseRows;
    if (gs > chunks) gs = int(chunks);
    if (gs < 1) gs = 1;
  }
  if (w == 1) slices = 2 * gs;   // the DMMA kernel writes its two row halves as separate slices
  int rc = ensureScratch(ctx, sizeof(T) * (kb * slices + kb));
  if (rc) return rc;
  T* out = reinterpret_cast<T*>(ctx->dScratch);
  T* partial = out + kb;
  if constexpr (w == 1) {
    auto ta = tableOf<double>(A), tx = tableOf<double>(X);
    double* part = reinterpret_cast<double*>(partial);
    const dim3 grid(gtiles, gs);
    const size_t smem = 128 + size_t(2) * (16 * ri + 16 * rj) * kDenseStride * sizeof(double);
#define MXG_GRAM(RI, RJ)                                                                                              \
  {                                                                                                                   \
    static bool attr = false;                                                                                         \
    if (!attr) {                                                                                                      \
      MXG_CUDA(cudaFuncSetAttribute(k_gram_mma<RI, RJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));     \
      attr = true;                                                                                                    \
    }                                                                                                                 \
    k_gram_mma<RI, RJ><<<grid, kDenseThreads, smem, ctx->stream>>>(ta, k, tx, b, A->ld, gtB, part);                    \
  }
    switch (ri * 4 + rj) {
      case 5: MXG_GRAM(1, 1); break;  case 6: MXG_GRAM(1, 2); break;  case 7: MXG_GRAM(1, 3); break;
      case 9: MXG_GRAM(2, 1); break;  case 10: MXG_GRAM(2, 2); break; case 11: MXG_GRAM(2, 3); break;
      case 13: MXG_GRAM(3, 1); break; case 14: MXG_GRAM(3, 2); break; default: MXG_GRAM(3, 3); break;
    }
#undef MXG_GRAM
  } else {
    k_trans_mv<T, KT, BT><<<dim3(tiles, slices), kBlock, 0, ctx->stream>>>(tableOf<T>(A), k, tableOf<T>(X), b, A->ld, tilesB, partial);
  }
  LAUNCH_CHECK(ctx);
  k_reduce_partials<T><<<int(kb), kBlock, 0, ctx->stream>>>(partial, slices, out);
  LAUNCH_CHECK(ctx);
  rc = allReduceScratch(ctx, kb * w);
  if (rc) return rc;
  std::vector<double> tmp(kb * w);
  rc = fetchScratch(ctx, tmp.data(), kb * w);
  if (rc) return rc;
  const T a = scalarOf<T>(alpha);
  T* Bt = reinterpret_cast<T*>(B);
  const T* src = reinterpret_cast<const T*>(tmp.data());
  for (int j = 0; j < b; ++j)
    for (int i = 0; i < k; ++i) Bt[i + size_t(j) * ldb] = a * src[i + size_t(j) * k];
  return MXG_OK;
}

template <class T>
int timesMatImpl(const double alpha[2], const mxg_mv* A, const double* B, int ldb, const double beta[2], mxg_mv* Y) {
  mxg_ctx* ctx = A->map->ctx;
  if (Y->ld == 0) return MXG_OK;
  constexpr int w = sizeof(T) / sizeof(double);
  constexpr int BT = (w == 1) ? 16 : 8;   // output columns per pass over A (accumulators stay in registers)
  constexpr int RT = 2;                     // rows per thread
  const int k = A->ncols, b = Y->ncols;
  const T al = scalarOf<T>(alpha), be = scalarOf<T>(beta);
  const bool useY = !isZero(be);
  if constexpr (w == 1) {
    if (k <= kUpdateMaxK) {
      // TMA-staged kernel: A is streamed once per block of <= 48 output columns
      for (int c0 = 0; c0 < b; c0 += 48) {
        const int cc = std::min(48, b - c0);
        std::vector<double> Bc(size_t(k) * cc);
        for (int j = 0; j < cc; ++j) std::memcpy(&Bc[size_t(j) * k], B + size_t(c0 + j) * ldb, sizeof(double) * k);
        MXG_CUDA(cudaMemcpyAsync(ctx->dDense, Bc.data(), Bc.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        const int rc_ = (cc + 15) / 16;
        const size_t k4 = size_t((k + 3) & ~3);
        const size_t smem = 128 + sizeof(double) * (((k4 * (16 * rc_ + 4) + 15) & ~size_t(15)) + size_t(2) * k4 * kDenseStride);
        const int64_t chunks = (Y->ld + kDenseRows - 1) / kDenseRows;
        const int grid = int(std::min<int64_t>(chunks, int64_t(ctx->numSMs) * 2));
        auto ta = tableOf<double>(A);
        auto ty = tableOf<double>(Y, c0, cc);
#define MXG_UPD(RC)                                                                                                    \
  {                                                                                                                    \
    static bool attr = false;                                                                                          \
    if (!attr) {                                                                                                       \
      MXG_CUDA(cudaFuncSetAttribute(k_update_mma<RC>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));        \
      attr = true;                                                                                                     \
    }                                                                                                                  \
    k_update_mma<RC><<<grid, kDenseThreads, smem, ctx->stream>>>(ta, k, ctx->dDense, cc, al, be, ty, Y->ld);            \
  }
        if (rc_ == 1) MXG_UPD(1) else if (rc_ == 2) MXG_UPD(2) else MXG_UPD(3)
#undef MXG_UPD
        LAUNCH_CHECK(ctx);
      }
      return MXG_OK;
    }
  }
  // columns of B that fit in one parameter block
  const int colsPerLaunch = kMaxBParam / (k * w);
  MXG_REQUIRE(colsPerLaunch >= 1, "mxg_mv_times_mat_add_mv: A has too many columns (%d) for one pass", k);
  const int grid = gridFor(ctx, Y->ld, kBlock * RT, 4);
  const size_t smem = sizeof(T) * size_t(k) * BT;
  for (int c0 = 0; c0 < b; c0 += colsPerLaunch) {
    const int cc = (b - c0 < colsPerLaunch) ? b - c0 : colsPerLaunch;
    DenseParam P;
    for (int j = 0; j < cc; ++j)
      std::memcpy(&P.v[size_t(j) * k * w], B + (size_t(c0 + j) * ldb) * w, sizeof(double) * k * w);
    // view of Y's columns c0..c0+cc
    ColTable<T> ty = tableOf<T>(Y, c0, cc);
    for (int j0 = 0; j0 < cc; j0 += BT) {
      const int bc = (cc - j0 < BT) ? cc - j0 : BT;
      k_times_mat<T, BT, RT><<<grid, kBlock, smem, ctx->stream>>>(tableOf<T>(A), k, P, j0, bc, al, be, useY, ty, Y->ld);
      LAUNCH_CHECK(ctx);
    }
  }
  return MXG_OK;
}

template <class T>
int removeConstImpl(mxg_mv* mv, int64_t count) {
  mxg_ctx* ctx = mv->map->ctx;
  const int nc = mv->ncols;
  constexpr int w = sizeof(T) / sizeof(double);
  int np = gridFor(ctx, mv->ld, kBlock * 8, 4);
  int cap = (ctx->numSMs * 4 + nc - 1) / nc;
  if (np > cap) np = cap;
  if (np < 1) np = 1;
  int rc = ensureScratch(ctx, sizeof(T) * (size_t(nc) * np + nc));
  if (rc) return rc;
  T* out = reinterpret_cast<T*>(ctx->dScratch);
  T* partial = out + nc;
  k_sum_partial<T><<<dim3(np, nc), kBlock, 0, ctx->stream>>>(tableOf<T>(mv), mv->ld, partial);
  LAUNCH_CHECK(ctx);
  k_reduce_partials<T><<<nc, kBlock, 0, ctx->stream>>>(partial, np, out);
  LAUNCH_CHECK(ctx);
  rc = allReduceScratch(ctx, size_t(nc) * w);
  if (rc) return rc;
  if (mv->ld > 0) {
    k_sub_mean<T><<<gridCols<T>(ctx, mv->ld, nc), kBlock, 0, ctx->stream>>>(tableOf<T>(mv), out, 1.0 / double(count), mv->ld);
    LAUNCH_CHECK(ctx);
  }
  return MXG_OK;
}

bool overlaps(const mxg_mv* a, const mxg_mv* b) {
  if (a->storage.get() != b->storage.get()) return false;
  for (void* pa : a->col)
    for (void* pb : b->col)
      if (pa == pb) return true;
  return false;
}

int checkSame(const char* fn, const mxg_mv* a, const mxg_mv* b, bool sameCols = true) {
  MXG_REQUIRE(a && b, "%s: NULL multivector", fn);
  MXG_REQUIRE(a->map->ctx == b->map->ctx, "%s: operands live on different contexts", fn);
  MXG_REQUIRE(a->ld == b->ld && a->map->nGlobal == b->map->nGlobal, "%s: operands have different maps", fn);
  MXG_REQUIRE(a->isComplex == b->isComplex, "%s: mixed real/complex operands", fn);
  if (sameCols) MXG_REQUIRE(a->ncols == b->ncols, "%s: column counts differ (%d vs %d)", fn, a->ncols, b->ncols);
  return MXG_OK;
}

}  // namespace

// Field output layout of MxIO::save (reference src/MxIO.cpp:166-221): a dense [cell][comp] array over the node grid, zero
// where the map holds no DOF. The global component index is comp + numComps * cell, so the dense index is the GID itself.
__global__ void k_scatter_grid(const double* __restrict__ x, int stride, const int64_t* __restrict__ gids, int64_t n,
                               int64_t lo, int64_t hi, double* __restrict__ outRe, double* __restrict__ outIm, int* err) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t g = gids[i];
    if (g < lo || g >= hi) { *err = 1; continue; }
    outRe[g - lo] = x[i * stride];
    if (stride == 2) outIm[g - lo] = x[i * 2 + 1];
  }
}

extern "C" {

int mxg_mv_fill(mxg_mv* mv, const double alpha[2]) {
  MXG_REQUIRE(mv && alpha, "mxg_mv_fill: NULL argument");
  MXG_CUDA(cudaSetDevice(mv->map->ctx->device));
  return mv->isComplex ? fillImpl<zd>(mv, alpha) : fillImpl<double>(mv, alpha);
}

int mxg_mv_scale(mxg_mv* mv, const double alpha[2]) {
  MXG_REQUIRE(mv && alpha, "mxg_mv_scale: NULL argument");
  MXG_CUDA(cudaSetDevice(mv->map->ctx->device));
  return mv->isComplex ? scaleColsImpl<zd>(mv, alpha, true) : scaleColsImpl<double>(mv, alpha, true);
}

int mxg_mv_scale_cols(mxg_mv* mv, const double* alphas) {
  MXG_REQUIRE(mv && alphas, "mxg_mv_scale_cols: NULL argument");
  MXG_CUDA(cudaSetDevice(mv->map->ctx->device));
  return mv->isComplex ? scaleColsImpl<zd>(mv, alphas, false) : scaleColsImpl<double>(mv, alphas, false);
}

int mxg_mv_conj(mxg_mv* mv) {
  MXG_REQUIRE(mv, "mxg_mv_conj: NULL argument");
  if (!mv->isComplex || mv->ld == 0) return MXG_OK;  // MxMultiVector.cpp:128-129: no-op for real
  mxg_ctx* ctx = mv->map->ctx;
  MXG_CUDA(cudaSetDevice(ctx->device));
  k_conj<<<gridCols<zd>(ctx, mv->ld, mv->ncols), kBlock, 0, ctx->stream>>>(tableOf<zd>(mv), mv->ld);
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}

int mxg_mv_random(mxg_mv* mv, uint64_t seed) {
  MXG_REQUIRE(mv, "mxg_mv_random: NULL argument");
  if (mv->ld == 0) return MXG_OK;
  mxg_ctx* ctx = mv->map->ctx;
  MXG_CUDA(cudaSetDevice(ctx->device));
  ColIds ids;
  for (int j = 0; j < mv->ncols; ++j) ids.v[j] = mv->baseCol[j];
  if (mv->isComplex)
    k_random_cplx<<<gridCols<zd>(ctx, mv->ld, mv->ncols), kBlock, 0, ctx->stream>>>(tableOf<zd>(mv), ids, mv->map->dGids, mv->ld, seed);
  else
    k_random_real<<<gridCols<double>(ctx, mv->ld, mv->ncols), kBlock, 0, ctx->stream>>>(tableOf<double>(mv), ids, mv->map->dGids, mv->ld, seed);
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}

int mxg_mv_add_mv(mxg_mv* dst, const double alpha[2], const mxg_mv* A, const double beta[2], const mxg_mv* B) {
  int rc = checkSame("mxg_mv_add_mv", dst, A);
  if (rc) return rc;
  rc = checkSame("mxg_mv_add_mv", dst, B);
  if (rc) return rc;
  MXG_REQUIRE(alpha && beta, "mxg_mv_add_mv: NULL scalar");
  MXG_CUDA(cudaSetDevice(dst->map->ctx->device));
  return dst->isComplex ? axpbyImpl<zd>(dst, alpha, A, beta, B) : axpbyImpl<double>(dst, alpha, A, beta, B);
}

// dst_j = alphas[j] * A_j + betas[j] * B_j: MvAddMv (MxAnasaziMV.cpp:89-111) with per-column scalars as in
// MvScale(vector) (MxAnasaziMV.hpp:110-118); A and/or B may alias dst.
int mxg_mv_axpby_cols(mxg_mv* dst, const double* alphas, const mxg_mv* A, const double* betas, const mxg_mv* B) {
  int rc = checkSame("mxg_mv_axpby_cols", dst, A);
  if (rc) return rc;
  rc = checkSame("mxg_mv_axpby_cols", dst, B);
  if (rc) return rc;
  MXG_REQUIRE(alphas && betas, "mxg_mv_axpby_cols: NULL scalar list");
  if (dst->ld == 0) return MXG_OK;
  mxg_ctx* ctx = dst->map->ctx;
  MXG_CUDA(cudaSetDevice(ctx->device));
  if (dst->isComplex) {
    ScalarList<zd> a, b;
    for (int j = 0; j < dst->ncols; ++j) { a.v[j] = {alphas[2 * j], alphas[2 * j + 1]}; b.v[j] = {betas[2 * j], betas[2 * j + 1]}; }
    k_axpby_cols<zd><<<gridCols<zd>(ctx, dst->ld, dst->ncols), kBlock, 0, ctx->stream>>>(tableOf<zd>(dst), a, tableOf<zd>(A), b, tableOf<zd>(B), dst->ld);
  } else {
    ScalarList<double> a, b;
    for (int j = 0; j < dst->ncols; ++j) { a.v[j] = alphas[j]; b.v[j] = betas[j]; }
    k_axpby_cols<double><<<gridCols<double>(ctx, dst->ld, dst->ncols), kBlock, 0, ctx->stream>>>(tableOf<double>(dst), a, tableOf<double>(A), b, tableOf<double>(B), dst->ld);
  }
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}

// removeConstField (MxGeoMultigridPrec.cpp:400-411, MxUtil.cpp:483-503): x_j -= (x_j . 1) / (1 . 1) 1, column by column;
// reduction, all-reduce and update are enqueued back to back, the sums never visit the host.
int mxg_mv_remove_const_field(mxg_mv* mv) {
  MXG_REQUIRE(mv, "mxg_mv_remove_const_field: NULL argument");
  MXG_CUDA(cudaSetDevice(mv->map->ctx->device));
  int64_t cnt = 0;
  int rc = mapGlobalCount(mv->map, &cnt);
  if (rc) return rc;
  MXG_REQUIRE(cnt > 0, "mxg_mv_remove_const_field: empty map");
  return mv->isComplex ? removeConstImpl<zd>(mv, cnt) : removeConstImpl<double>(mv, cnt);
}

// MxGridField::zeroUnusedComponents (MxGridField.cpp:548-576, called on the initial block at MxSolver.cpp:65): zero the
// entries whose shape fraction is 0. fracs: one-column multivector on the same map holding the fractions (real part used).
int mxg_mv_zero_unused(mxg_mv* mv, const mxg_mv* fracs) {
  MXG_REQUIRE(mv && fracs, "mxg_mv_zero_unused: NULL argument");
  MXG_REQUIRE(fracs->ncols >= 1 && fracs->ld == mv->ld && fracs->map->ctx == mv->map->ctx, "mxg_mv_zero_unused: fraction vector does not match");
  if (mv->ld == 0) return MXG_OK;
  mxg_ctx* ctx = mv->map->ctx;
  MXG_CUDA(cudaSetDevice(ctx->device));
  const double* f = static_cast<const double*>(fracs->col[0]);
  const int fs = fracs->isComplex ? 2 : 1;
  if (mv->isComplex) k_zero_unused<zd><<<gridCols<zd>(ctx, mv->ld, mv->ncols), kBlock, 0, ctx->stream>>>(tableOf<zd>(mv), f, fs, mv->ld);
  else k_zero_unused<double><<<gridCols<double>(ctx, mv->ld, mv->ncols), kBlock, 0, ctx->stream>>>(tableOf<double>(mv), f, fs, mv->ld);
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}

int mxg_mv_update(mxg_mv* dst, const double a[2], const mxg_mv* A, const double s[2]) {
  return mxg_mv_add_mv(dst, a, A, s, dst);
}

int mxg_mv_assign(mxg_mv* dst, const mxg_mv* src) {
  int rc = checkSame("mxg_mv_assign", dst, src);
  if (rc) return rc;
  if (dst->ld == 0) return MXG_OK;
  mxg_ctx* ctx = dst->map->ctx;
  MXG_CUDA(cudaSetDevice(ctx->device));
  if (dst->isComplex)
    k_copy<zd><<<gridCols<zd>(ctx, dst->ld, dst->ncols), kBlock, 0, ctx->stream>>>(tableOf<zd>(dst), tableOf<zd>(src), dst->ld);
  else
    k_copy<double><<<gridCols<double>(ctx, dst->ld, dst->ncols), kBlock, 0, ctx->stream>>>(tableOf<double>(dst), tableOf<double>(src), dst->ld);
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}

int mxg_mv_set_block(mxg_mv* dst, const mxg_mv* src, const int* index, int n) {
  int rc = checkSame("mxg_mv_set_block", dst, src, false);
  if (rc) return rc;
  MXG_REQUIRE(index && n >= 1 && n <= src->ncols, "mxg_mv_set_block: bad index list");
  for (int j = 0; j < n; ++j)
    MXG_REQUIRE(index[j] >= 0 && index[j] < dst->ncols, "mxg_mv_set_block: index %d out of range", index[j]);
  std::vector<int> cols(index, index + n);
  mxg_mv* view = nullptr;
  rc = mxg_mv_view(dst, cols.data(), n, &view);
  if (rc) return rc;
  mxg_mv* sview = nullptr;
  std::vector<int> first(n);
  for (int j = 0; j < n; ++j) first[j] = j;
  rc = mxg_mv_view(const_cast<mxg_mv*>(src), first.data(), n, &sview);
  if (rc == MXG_OK) rc = mxg_mv_assign(view, sview);
  if (sview) mxg_mv_destroy(sview);
  mxg_mv_destroy(view);
  return rc;
}

int mxg_mv_dot(const mxg_mv* a, const mxg_mv* b, double* out) {
  int rc = checkSame("mxg_mv_dot", a, b);
  if (rc) return rc;
  MXG_REQUIRE(out, "mxg_mv_dot: out is NULL");
  mxg_ctx* ctx = a->map->ctx;
  MXG_CUDA(cudaSetDevice(ctx->device));
  rc = a->isComplex ? dotToScratch<zd>(a, b) : dotToScratch<double>(a, b);
  if (rc) return rc;
  return fetchScratch(ctx, out, size_t(a->ncols) * (a->isComplex ? 2 : 1));
}

int mxg_mv_norm2(const mxg_mv* mv, double* out) {
  MXG_REQUIRE(mv && out, "mxg_mv_norm2: NULL argument");
  mxg_ctx* ctx = mv->map->ctx;
  MXG_CUDA(cudaSetDevice(ctx->device));
  int rc = mv->isComplex ? dotToScratch<zd>(mv, mv) : dotToScratch<double>(mv, mv);
  if (rc) return rc;
  const int w = mv->isComplex ? 2 : 1;
  std::vector<double> tmp(size_t(mv->ncols) * w);
  rc = fetchScratch(ctx, tmp.data(), tmp.size());
  if (rc) return rc;
  for (int j = 0; j < mv->ncols; ++j) out[j] = std::sqrt(tmp[size_t(j) * w]);
  return MXG_OK;
}

int mxg_mv_normalize(mxg_mv* mv) {
  MXG_REQUIRE(mv, "mxg_mv_normalize: NULL argument");
  std::vector<double> nrm(mv->ncols);
  int rc = mxg_mv_norm2(mv, nrm.data());
  if (rc) return rc;
  const int w = mv->isComplex ? 2 : 1;
  std::vector<double> inv(size_t(mv->ncols) * w, 0.0);
  for (int j = 0; j < mv->ncols; ++j) inv[size_t(j) * w] = nrm[j] > 0 ? 1.0 / nrm[j] : 0.0;
  return mxg_mv_scale_cols(mv, inv.data());
}

int mxg_mv_trans_mv(const double alpha[2], const mxg_mv* A, const mxg_mv* X, double* B, int ldb) {
  int rc = checkSame("mxg_mv_trans_mv", A, X, false);
  if (rc) return rc;
  MXG_REQUIRE(alpha && B && ldb >= A->ncols, "mxg_mv_trans_mv: bad B / ldb (need ldb >= %d)", A->ncols);
  MXG_CUDA(cudaSetDevice(A->map->ctx->device));
  return A->isComplex ? transMvImpl<zd>(alpha, A, X, B, ldb) : transMvImpl<double>(alpha, A, X, B, ldb);
}

int mxg_mv_times_mat_add_mv(const double alpha[2], const mxg_mv* A, const double* B, int ldb, const double beta[2], mxg_mv* Y) {
  int rc = checkSame("mxg_mv_times_mat_add_mv", A, Y, false);
  if (rc) return rc;
  MXG_REQUIRE(alpha && beta && B && ldb >= A->ncols, "mxg_mv_times_mat_add_mv: bad B / ldb (need ldb >= %d)", A->ncols);
  // Y may share columns with A (in-place right-multiplication of a basis block) on the TMA-staged real kernel, which holds
  // a row chunk of A completely in shared memory before it writes those rows; otherwise the operands must be disjoint
  const bool inPlaceOk = !A->isComplex && A->ncols <= kUpdateMaxK && Y->ncols <= 48;
  MXG_REQUIRE(inPlaceOk || !overlaps(A, Y), "mxg_mv_times_mat_add_mv: A and Y must not share columns (complex, > %d source or > 48 result columns)", kUpdateMaxK);
  MXG_CUDA(cudaSetDevice(A->map->ctx->device));
  return A->isComplex ? timesMatImpl<zd>(alpha, A, B, ldb, beta, Y) : timesMatImpl<double>(alpha, A, B, ldb, beta, Y);
}

int mxg_mv_to_grid(const mxg_mv* mv, int col, int64_t gid_lo, int64_t gid_hi, double* out_real, double* out_imag) {
  MXG_REQUIRE(mv && out_real, "mxg_mv_to_grid: NULL argument");
  MXG_REQUIRE(col >= 0 && col < mv->ncols, "mxg_mv_to_grid: column %d out of range (%d columns)", col, mv->ncols);
  MXG_REQUIRE(gid_hi >= gid_lo, "mxg_mv_to_grid: empty or reversed GID range");
  MXG_REQUIRE(!mv->isComplex || out_imag, "mxg_mv_to_grid: complex field needs out_imag");
  mxg_ctx* ctx = mv->map->ctx;
  MXG_CUDA(cudaSetDevice(ctx->device));
  const int64_t len = gid_hi - gid_lo, n = mv->ld;
  if (len == 0) { MXG_REQUIRE(n == 0, "mxg_mv_to_grid: owned DOFs outside the GID range"); return MXG_OK; }
  const int parts = mv->isComplex ? 2 : 1;
  double* dOut = nullptr;
  int* dErr = nullptr;
  MXG_CUDA(cudaMalloc(&dOut, size_t(len) * parts * sizeof(double) + sizeof(int)));
  dErr = reinterpret_cast<int*>(dOut + size_t(len) * parts);
  cudaError_t e = cudaMemsetAsync(dOut, 0, size_t(len) * parts * sizeof(double) + sizeof(int), ctx->stream);
  if (e == cudaSuccess && n > 0) {
    const int blocks = int(std::min<int64_t>((n + 255) / 256, int64_t(ctx->numSMs) * 8));
    k_scatter_grid<<<blocks, 256, 0, ctx->stream>>>(static_cast<const double*>(mv->col[col]), parts, mv->map->dGids, n, gid_lo, gid_hi,
                                                    dOut, dOut + len, dErr);
    ++ctx->launches;
    e = cudaGetLastError();
  }
  int hErr = 0;
  if (e == cudaSuccess) e = cudaMemcpyAsync(out_real, dOut, size_t(len) * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess && mv->isComplex)
    e = cudaMemcpyAsync(out_imag, dOut + len, size_t(len) * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(&hErr, dErr, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFree(dOut);
  MXG_REQUIRE(e == cudaSuccess, "mxg_mv_to_grid: %s", cudaGetErrorString(e));
  MXG_REQUIRE(hErr == 0, "mxg_mv_to_grid: owned DOFs outside the GID range [%lld, %lld)", (long long)gid_lo, (long long)gid_hi);
  return MXG_OK;
}

}  // extern "C"
