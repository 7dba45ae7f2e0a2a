// Exclusive prefix scan of int32 counts into int64 offsets (three passes: chunk totals, scan of the totals in one
// block, scan inside every chunk). Set-up code of the operator assembly and of the layout builder.
#pragma once
#include <algorithm>

#include "mxg_internal.h"

namespace mxg {

constexpr int kScanBlock = 256;
constexpr int kScanChunk = 2048;    // items per block (8 per thread)

// pass 1: per-chunk totals
static __global__ void __launch_bounds__(kScanBlock) k_scan_sums(const int32_t* __restrict__ in, int64_t n, int64_t* __restrict__ sums) {
  __shared__ int64_t sh[kScanBlock];
  const int64_t base = int64_t(blockIdx.x) * kScanChunk;
  int64_t s = 0;
  for (int k = 0; k < kScanChunk / kScanBlock; ++k) {
    const int64_t i = base + int64_t(k) * kScanBlock + threadIdx.x;
    if (i < n) s += in[i];
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = kScanBlock / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) sums[blockIdx.x] = sh[0];
}
// pass 2: exclusive scan of the chunk totals in one block (a running carry over tiles of kScanBlock totals)
static __global__ void __launch_bounds__(kScanBlock) k_scan_chunks(int64_t* __restrict__ sums, int64_t numChunks, int64_t* __restrict__ total) {
  __shared__ int64_t sh[kScanBlock];
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t tile = 0; tile < numChunks; tile += kScanBlock) {
    const int64_t i = tile + threadIdx.x;
    const int64_t v = i < numChunks ? sums[i] : 0;
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < kScanBlock; o <<= 1) {       // inclusive Hillis-Steele
      const int64_t t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
      __syncthreads();
      sh[threadIdx.x] += t;
      __syncthreads();
    }
    if (i < numChunks) sums[i] = carry + sh[threadIdx.x] - v;
    __syncthreads();
    if (threadIdx.x == kScanBlock - 1) carry += sh[kScanBlock - 1];
    __syncthreads();
  }
  if (threadIdx.x == 0) *total = carry;
}
// pass 3: exclusive scan inside every chunk, offset by the chunk's start; thread t owns 8 consecutive items
static __global__ void __launch_bounds__(kScanBlock) k_scan_write(const int32_t* __restrict__ in, int64_t n, const int64_t* __restrict__ sums,
                                                          const int64_t* __restrict__ total, int64_t* __restrict__ out) {
  __shared__ int64_t sh[kScanBlock];
  constexpr int per = kScanChunk / kScanBlock;
  const int64_t first = int64_t(blockIdx.x) * kScanChunk + int64_t(threadIdx.x) * per;
  int32_t v[per];
  int64_t s = 0;
  for (int k = 0; k < per; ++k) {
    v[k] = first + k < n ? in[first + k] : 0;
    s += v[k];
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 1; o < kScanBlock; o <<= 1) {
    const int64_t t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
    __syncthreads();
    sh[threadIdx.x] += t;
    __syncthreads();
  }
  int64_t run = sums[blockIdx.x] + sh[threadIdx.x] - s;
  for (int k = 0; k < per; ++k) {
    if (first + k < n) out[first + k] = run;
    run += v[k];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = *total;
}


// out[0..n] = exclusive scan of in[0..n-1] (out[n] = total); the total also lands in *total after a stream synchronise
inline cudaError_t exclusiveScan(mxg_ctx* ctx, const int32_t* in, int64_t* out, int64_t n, int64_t* total) {
  const int64_t chunks = std::max<int64_t>((n + kScanChunk - 1) / kScanChunk, 1);
  int64_t* sums = nullptr;
  cudaError_t e = cudaMalloc(&sums, size_t(chunks + 1) * sizeof(int64_t));
  if (e != cudaSuccess) return e;
  k_scan_sums<<<unsigned(chunks), kScanBlock, 0, ctx->stream>>>(in, n, sums);
  k_scan_chunks<<<1, kScanBlock, 0, ctx->stream>>>(sums, chunks, sums + chunks);
  k_scan_write<<<unsigned(chunks), kScanBlock, 0, ctx->stream>>>(in, n, sums, sums + chunks, out);
  ctx->launches += 3;
  e = cudaGetLastError();
  if (e == cudaSuccess && total) e = cudaMemcpyAsync(total, sums + chunks, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFree(sums);
  return e;
}

}  // namespace mxg
