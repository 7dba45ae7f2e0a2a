// Operator assembly on the device (SURVEY 8 f2, f3; include/mxasm.h): cut-cell fractions of a CSG shape, DOF maps,
// the Yee operator generators and the CRS products / sums that chain them into curlCurl, gradDiv, vecLapl and scaLapl,
// one thread per cell or per operator row. The arithmetic lives in mxg_yee.h / mxg_shape.h (host/device code, replayed on
// the CPU by the tests); this file supplies the CUDA executor: kernels, a three-pass prefix scan, memory.
//
// This translation unit is compiled with -fmad=false: the reference's host code rounds a*b+c twice, and the generated
// matrices have to carry the very same doubles for the SpMV parity gate to hold downstream.
#include <algorithm>
#include <cstring>
#include <string>
#include <unordered_map>

#include "mxasm.h"
#include "mxg_internal.h"
#include "mxg_asm_impl.h"
#include "mxg_scan.cuh"
#include "mxg_shape.h"

namespace {

constexpr int kAsmBlock = 256;

template <class F>
__global__ void __launch_bounds__(kAsmBlock) k_asm_rows(int64_t n, F f) {
  for (int64_t i = int64_t(blockIdx.x) * kAsmBlock + threadIdx.x; i < n; i += int64_t(gridDim.x) * kAsmBlock) f(i);
}

__global__ void __launch_bounds__(kAsmBlock) k_asm_max(const int32_t* __restrict__ in, int64_t n, int* __restrict__ out) {
  int m = 0;
  for (int64_t i = int64_t(blockIdx.x) * kAsmBlock + threadIdx.x; i < n; i += int64_t(gridDim.x) * kAsmBlock) m = max(m, in[i]);
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(out, m);
}

[[noreturn]] void fail(const char* what, cudaError_t e) {
  throw std::runtime_error(std::string(what) + ": " + cudaGetErrorString(e));
}

struct DeviceExec {
  mxg_ctx* ctx;
  std::unordered_map<void*, size_t> sizes;   // live allocations, counted into ctx->asmBytes / asmPeak
  explicit DeviceExec(mxg_ctx* c) : ctx(c) {
    if (!c) throw std::runtime_error("operator assembly needs a context (mxg_ctx_create)");
    cudaSetDevice(c->device);
  }
  template <class T>
  T* alloc(int64_t n) {
    void* p = nullptr;
    const size_t bytes = size_t(n > 0 ? n : 1) * sizeof(T);
    const cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) fail("device allocation of the operator assembly", e);
    sizes[p] = bytes;
    ctx->asmBytes += int64_t(bytes);
    ctx->asmPeak = std::max(ctx->asmPeak, ctx->asmBytes);
    return static_cast<T*>(p);
  }
  void free(void* p) {
    if (!p) return;
    const auto it = sizes.find(p);
    if (it != sizes.end()) {
      ctx->asmBytes -= int64_t(it->second);
      sizes.erase(it);
    }
    cudaFree(p);
  }
  void check(const char* what) {
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) fail(what, e);
  }
  template <class F>
  void forEach(int64_t n, const F& f) {
    static_assert(sizeof(F) <= 3072, "row functor too large for a kernel parameter block");
    if (n <= 0) return;
    const int64_t blocks = std::min<int64_t>((n + kAsmBlock - 1) / kAsmBlock, int64_t(1) << 30);
    k_asm_rows<F><<<unsigned(blocks), kAsmBlock, 0, ctx->stream>>>(n, f);
    ctx->launches++;
    check("assembly kernel launch");
  }
  int64_t scan(const int32_t* in, int64_t* out, int64_t n) {
    int64_t total = 0;
    const cudaError_t e = mxg::exclusiveScan(ctx, in, out, n, &total);
    if (e != cudaSuccess) fail("prefix scan of the operator assembly", e);
    return total;
  }
  int maxOf(const int32_t* in, int64_t n) {
    int* d = alloc<int>(1);
    cudaMemsetAsync(d, 0, sizeof(int), ctx->stream);
    const int64_t blocks = std::min<int64_t>((n + kAsmBlock - 1) / kAsmBlock, 4096);
    if (n > 0) {
      k_asm_max<<<unsigned(blocks), kAsmBlock, 0, ctx->stream>>>(in, n, d);
      ctx->launches++;
    }
    check("row maximum launch");
    int m = 0;
    toHost(&m, d, sizeof(int));
    free(d);
    return m;
  }
  void toHost(void* dst, const void* src, size_t bytes) {
    if (!bytes) return;
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) fail("device -> host copy of the operator assembly", e);
  }
  void toExec(void* dst, const void* src, size_t bytes) {
    if (!bytes) return;
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);   // the source may be a stack temporary
    if (e != cudaSuccess) fail("host -> device copy of the operator assembly", e);
  }
  void zero(void* p, size_t bytes) {
    if (!bytes) return;
    const cudaError_t e = cudaMemsetAsync(p, 0, bytes, ctx->stream);
    if (e != cudaSuccess) fail("device memset of the operator assembly", e);
  }
  void sync() {
    const cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) fail("operator assembly", e);
  }
};

}  // namespace

#define MXA_FN(name) mxg_##name
#define MXA_EXEC DeviceExec
#define MXA_CTX mxg_ctx
#define MXA_SIM_T mxg_sim
#define MXA_DCSR_T mxg_dcsr
#define MXA_SHAPE_T mxg_shape
#define MXA_NEW_EXEC(ctx) (new DeviceExec(ctx))
#define MXA_FAIL(code, msg)        \
  do {                             \
    mxg::setError("%s", (msg));    \
    return (code);                 \
  } while (0)

#include "mxg_asm_api.inc"

extern "C" {

// MxCrsMatrix::fillComplete for an operator assembled on the device (MxCrsMatrix.cpp:325-342): the rows this rank's
// row map owns become a device operator (pattern dictionary / sliced ELL, halo plan) without the host ever seeing
// them: the layout is built by kernels too (mxg::crsCreateFromDevice). A domain map that is not a run of the column
// field map, and ordered maps, take the host CSR route instead: the rows are downloaded and mxg_crs_create_opts lays
// them out with the same kernels.
int mxg_crs_create_from_dcsr(mxg_map* row_map, mxg_map* domain_map, const mxg_dcsr* a, int layout, mxg_crs** out) {
  const CsrHandle* A = reinterpret_cast<const CsrHandle*>(a);
  MXG_REQUIRE(row_map && domain_map && A && out, "mxg_crs_create_from_dcsr: NULL argument");
  const int rf = A->rowField(), cf = A->colField();
  MXG_REQUIRE(rf >= 0 && cf >= 0, "mxg_crs_create_from_dcsr: the matrix does not know which fields its rows and columns live on");
  try {
    mxa::Assembler<DeviceExec>& asR = *A->rows()->as;
    mxa::Assembler<DeviceExec>& asC = *A->cols()->as;
    MXG_REQUIRE(domain_map->nGlobal == asC.numGlobal(cf) && row_map->nGlobal == asR.numGlobal(rf),
                "mxg_crs_create_from_dcsr: maps do not span the simulation's GID space");
    MXG_REQUIRE(asR.mapSize(rf) == A->mapRows() && asC.mapSize(cf) == A->ncols(), "mxg_crs_create_from_dcsr: the matrix does not live on these field maps");
    std::vector<int64_t> rowG(static_cast<size_t>(asR.mapSize(rf)), 0), colG(static_cast<size_t>(asC.mapSize(cf)), 0);
    asR.copyMap(rf, rowG.data());
    asC.copyMap(cf, colG.data());
    // the rank's rows: one contiguous run of the field map (x-slabs)
    int64_t r0 = 0, r1 = 0;
    if (row_map->nLocal > 0) {
      r0 = int64_t(std::lower_bound(rowG.begin(), rowG.end(), row_map->gids.front()) - rowG.begin());
      r1 = r0 + row_map->nLocal;
      MXG_REQUIRE(r1 <= int64_t(rowG.size()) && std::memcmp(rowG.data() + r0, row_map->gids.data(), size_t(row_map->nLocal) * sizeof(int64_t)) == 0,
                  "mxg_crs_create_from_dcsr: the row map is not a contiguous run of the simulation's %s map",
                  rf == mxy::FIELD_B ? "B" : (rf == mxy::FIELD_E ? "E" : "psi"));
    }
    // ... which the matrix must store (a slab operator from mxg_sim_op_rows stores its rows only)
    const int64_t s0 = r0 - A->rowBegin();
    MXG_REQUIRE(r1 == r0 || (s0 >= 0 && s0 + (r1 - r0) <= A->nrows()),
                "mxg_crs_create_from_dcsr: the matrix stores the rows [%lld, %lld) of its map, not the row map's [%lld, %lld)",
                (long long)A->rowBegin(), (long long)(A->rowBegin() + A->nrows()), (long long)r0, (long long)r1);
    // this rank's columns: the run of the column field map its domain map owns
    int64_t c0 = 0;
    bool domIsRun = true;
    if (domain_map->nLocal > 0) {
      c0 = int64_t(std::lower_bound(colG.begin(), colG.end(), domain_map->gids.front()) - colG.begin());
      domIsRun = c0 + domain_map->nLocal <= int64_t(colG.size()) &&
                 std::memcmp(colG.data() + c0, domain_map->gids.data(), size_t(domain_map->nLocal) * sizeof(int64_t)) == 0;
    }
    if (domIsRun && row_map->perm.empty() && domain_map->perm.empty()) {
      const int64_t* rp = (A->isComplex ? A->c.rowptr : A->r.rowptr) + (r1 > r0 ? s0 : 0);
      const int32_t* col = A->isComplex ? A->c.col : A->r.col;
      const void* val = A->isComplex ? static_cast<const void*>(A->c.val) : static_cast<const void*>(A->r.val);
      return mxg::crsCreateFromDevice(row_map, domain_map, rp, col, val, c0, int64_t(colG.size()), colG.data(), A->isComplex, layout, out);
    }
    // maps the device front end does not take: the rows pass through the host CSR entry point
    const int64_t n = r1 - r0;
    std::vector<int64_t> rowptr(static_cast<size_t>(n) + 1, 0);
    const int64_t d0 = r1 > r0 ? s0 : 0;
    int rc = mxg_dcsr_download(a, d0, d0 + n, rowptr.data(), nullptr, nullptr);
    if (rc) return rc;
    const int64_t cnt = rowptr[size_t(n)];
    std::vector<int32_t> col(static_cast<size_t>(std::max<int64_t>(cnt, 1)), 0);
    std::vector<double> val(static_cast<size_t>(std::max<int64_t>(cnt, 1)) * (A->isComplex ? 2 : 1), 0.0);
    rc = mxg_dcsr_download(a, d0, d0 + n, rowptr.data(), col.data(), val.data());
    if (rc) return rc;
    std::vector<int64_t> gcol(static_cast<size_t>(std::max<int64_t>(cnt, 1)), 0);
    for (int64_t q = 0; q < cnt; ++q) gcol[size_t(q)] = colG[size_t(col[size_t(q)])];
    std::vector<int32_t>().swap(col);
    return mxg_crs_create_opts(row_map, domain_map, rowptr.data(), gcol.data(), val.data(), A->isComplex, layout, out);
  } catch (const std::exception& e) {
    MXG_REQUIRE(false, "mxg_crs_create_from_dcsr: %s", e.what());
  }
}

// The DOF map of a field as an mxg_map of this context: the rows [begin, end) of the field's map (an x-slab when the
// caller cuts at plane boundaries), or the whole map with begin = 0, end = -1.
int mxg_sim_make_map(mxg_sim* sim, const char* field, int64_t begin, int64_t end, mxg_map** out) {
  SimHandle* h = reinterpret_cast<SimHandle*>(sim);
  const int k = fieldIndex(field);
  MXG_REQUIRE(h && k >= 0 && out, "mxg_sim_make_map: bad argument");
  MXG_REQUIRE(h->as->isSetUp(), "mxg_sim_make_map: call mxg_sim_setup first");
  try {
    const int64_t n = h->as->mapSize(k);
    if (end < 0) end = n;
    MXG_REQUIRE(begin >= 0 && begin <= end && end <= n, "mxg_sim_make_map: range outside the map");
    std::vector<int64_t> g(static_cast<size_t>(n), 0);
    h->as->copyMap(k, g.data());
    return mxg_map_create(h->ctx, h->as->numGlobal(k), g.data() + begin, end - begin, out);
  } catch (const std::exception& e) {
    MXG_REQUIRE(false, "mxg_sim_make_map: %s", e.what());
  }
}

// Device bytes the assembly executors of a context hold now (out[0]) and at most since the last reset (out[1]):
// simulations (fractions, maps), matrices and the temporaries of the passes. reset_peak != 0 restarts the peak at the
// current value.
int mxg_asm_memory(mxg_ctx* ctx, int64_t out[2], int reset_peak) {
  MXG_REQUIRE(ctx && out, "mxg_asm_memory: NULL argument");
  if (reset_peak) ctx->asmPeak = ctx->asmBytes;
  out[0] = ctx->asmBytes;
  out[1] = ctx->asmPeak;
  return 0;
}

}  // extern "C"
