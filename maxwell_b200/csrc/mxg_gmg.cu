// libmxgpu: geometric multigrid preconditioner on the GPU (K15-K19 of SURVEY.md section 2.3).
//
// Semantic spec: MxGeoMultigridPrec (reference src/MxGeoMultigridPrec.cpp) -- dead code in the
// reference (commented out of its build), so this follows its structure, not its numbers:
//   setup       :98-240   per-level smoothers; Chebyshev with eigenvalue ratio 30 and lambda_max
//                         of D^-1 A estimated iteratively (:199-216)
//   vCycle      :243-398  smooth, r = b - A x (:312-314), coarsen (:325), recurse, refine + add
//                         (:345-350), smooth (:375)
//   fullVCycle  :547-616  coarsen b to all levels, coarse solve, then refine + `cycles` V-cycles
//                         per level on the way up
//   ApplyInverse:496-542
// Level operators, restriction and prolongation are ordinary mxg_crs handles (re-discretised
// operators and trilinear field interpolators generated on the host), so every SpMM below is
// the pattern-compressed kernel of mxg_spmv.cu and works unchanged on several ranks.
// The coarse direct solve (Ifpack_Amesos/KLU, :158-181) is replaced by a high-degree Chebyshev
// sweep on the coarsest level, which stays on the GPU and is deterministic.
#include <cmath>
#include <cstring>

#include "mxg_internal.h"

using namespace mxg;

struct mxg_gmg {
  mxg_ctx* ctx = nullptr;
  int nlevels = 0;
  bool isComplex = false;
  mxg_gmg_params prm{};
  std::vector<const mxg_crs*> A, R, P;
  std::vector<double> lambdaMax;
  // per-level work vectors (x, b, v = A x / residual, w = Chebyshev direction), sized lazily
  std::vector<mxg_mv*> x, b, v, w;
  int workCols = 0;
  int64_t spmmCount = 0;
};

namespace {

constexpr int kBlock = 256;

#define LAUNCH_CHECK(ctx)         \
  do {                            \
    (ctx)->launches++;            \
    MXG_CUDA(cudaGetLastError()); \
  } while (0)

__device__ __forceinline__ double mulD(double d, double a) { return d * a; }
__device__ __forceinline__ zd mulD(zd d, zd a) { return d * a; }
__device__ __forceinline__ double scaleR(double s, double a) { return s * a; }
__device__ __forceinline__ zd scaleR(double s, zd a) { return {s * a.x, s * a.y}; }

// Chebyshev step: W = c1*W + c2 * Dinv .* (B - V);  X += W.   first: W = c2 * Dinv .* (B - V)
// zeroStart (V not formed, X = 0):                     W = c2 * Dinv .* B;  X = W
template <class T>
__global__ void __launch_bounds__(kBlock) k_cheb(ColTable<T> W, ColTable<T> X, ColTable<T> B, ColTable<T> V,
                                                 const T* __restrict__ dinv, double c1, double c2, int mode, int64_t n) {
  T* __restrict__ w = W.p[blockIdx.y];
  T* __restrict__ x = X.p[blockIdx.y];
  const T* __restrict__ b = B.p[blockIdx.y];
  const T* __restrict__ v = V.p[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock) {
    const T d = dinv[i];
    if (mode == 2) {  // zero start
      const T wn = scaleR(c2, mulD(d, b[i]));
      w[i] = wn;
      x[i] = wn;
    } else {
      T wn = scaleR(c2, mulD(d, b[i] - v[i]));
      if (mode == 0) wn = wn + scaleR(c1, w[i]);
      w[i] = wn;
      x[i] = x[i] + wn;
    }
  }
}

template <class T>
__global__ void __launch_bounds__(kBlock) k_diag_scale(ColTable<T> Y, ColTable<T> Xs, const T* __restrict__ d, int64_t n) {
  T* __restrict__ y = Y.p[blockIdx.y];
  const T* __restrict__ x = Xs.p[blockIdx.y];
  for (int64_t i = blockIdx.x * int64_t(kBlock) + threadIdx.x; i < n; i += int64_t(gridDim.x) * kBlock) y[i] = mulD(d[i], x[i]);
}

dim3 gridCols(const mxg_ctx* ctx, int64_t n, int ncols) {
  int perCol = gridFor(ctx, n, kBlock * 4, 8);
  int cap = (ctx->numSMs * 8 + ncols - 1) / ncols;
  if (perCol > cap) perCol = cap;
  if (perCol < 1) perCol = 1;
  return dim3(perCol, ncols);
}

template <class T>
int chebLaunch(mxg_gmg* g, int l, mxg_mv* x, const mxg_mv* b, double c1, double c2, int mode) {
  mxg_ctx* ctx = g->ctx;
  const int64_t n = g->A[l]->nRows;
  if (n == 0) return MXG_OK;
  const int nc = x->ncols;
  // views of the level work vectors restricted to nc columns
  k_cheb<T><<<gridCols(ctx, n, nc), kBlock, 0, ctx->stream>>>(tableOf<T>(g->w[l], 0, nc), tableOf<T>(x), tableOf<T>(b),
                                                              tableOf<T>(g->v[l], 0, nc), static_cast<const T*>(g->A[l]->dInvDiag),
                                                              c1, c2, mode, n);
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}

int viewCols(mxg_mv* parent, int nc, mxg_mv** out) {
  std::vector<int> cols(nc);
  for (int j = 0; j < nc; ++j) cols[j] = j;
  return mxg_mv_view(parent, cols.data(), nc, out);
}

// Chebyshev smoother of the given degree on D^-1 A over [lmax/ratio, 1.1*lmax] (Ifpack_Chebyshev
// recurrence; the smoother named in MxGeoMultigridPrec.cpp:110-122).
template <class T>
int smooth(mxg_gmg* g, int l, mxg_mv* x, const mxg_mv* b, int degree, double ratio, bool zeroStart) {
  if (degree <= 0) return MXG_OK;
  const double lmax = g->lambdaMax[l];
  const double alpha = lmax / ratio, beta = 1.1 * lmax;
  const double delta = 2.0 / (beta - alpha), theta = 0.5 * (beta + alpha), s1 = theta * delta;
  const int nc = x->ncols;
  mxg_mv* vview = nullptr;
  int rc = viewCols(g->v[l], nc, &vview);
  if (rc) return rc;
  auto applyA = [&]() {
    g->spmmCount++;
    return mxg_crs_apply(g->A[l], x, vview);
  };
  if (zeroStart) {
    rc = chebLaunch<T>(g, l, x, b, 0.0, 1.0 / theta, 2);
  } else {
    rc = applyA();
    if (!rc) rc = chebLaunch<T>(g, l, x, b, 0.0, 1.0 / theta, 1);
  }
  double rhok = 1.0 / s1;
  for (int k = 1; k < degree && !rc; ++k) {
    rc = applyA();
    const double rhokp1 = 1.0 / (2.0 * s1 - rhok);
    const double c1 = rhokp1 * rhok, c2 = 2.0 * rhokp1 * delta;
    rhok = rhokp1;
    if (!rc) rc = chebLaunch<T>(g, l, x, b, c1, c2, 0);
  }
  mxg_mv_destroy(vview);
  return rc;
}

template <class T>
int vcycle(mxg_gmg* g, int l, mxg_mv* x, const mxg_mv* b, bool zeroStart) {
  const mxg_gmg_params& p = g->prm;
  if (l == g->nlevels - 1)
    return smooth<T>(g, l, x, b, g->nlevels == 1 ? p.smoother_degree : p.coarse_degree,
                     g->nlevels == 1 ? p.eig_ratio : p.coarse_eig_ratio, zeroStart);
  int rc = smooth<T>(g, l, x, b, p.smoother_degree, p.eig_ratio, zeroStart);
  if (rc) return rc;
  const int nc = x->ncols;
  mxg_mv *r = nullptr, *bc = nullptr, *xc = nullptr;
  if ((rc = viewCols(g->v[l], nc, &r))) return rc;
  if ((rc = viewCols(g->b[l + 1], nc, &bc))) { mxg_mv_destroy(r); return rc; }
  if ((rc = viewCols(g->x[l + 1], nc, &xc))) { mxg_mv_destroy(r); mxg_mv_destroy(bc); return rc; }
  const double one[2] = {1, 0}, mone[2] = {-1, 0};
  // r = b - A x  (fused SpMM epilogue)
  rc = mxg_mv_assign(r, b);
  if (!rc) { g->spmmCount++; rc = mxg_crs_apply_axpby(g->A[l], mone, x, one, r); }
  // coarsen (MxGeoMultigridPrec.cpp:447-452). With "remove const field" the fine residual is projected before it is
  // restricted, as are the restricted right-hand side and the correction below. With Q = I - 1 1^T / n the coarse-grid
  // correction is then Q P C R Q with R = P^T / 8, which is symmetric, and so is the cycle that block CG runs on. Projecting
  // only bc and the correction gives Q P C Q_c R, which is not. (P maps the coarse constant to the fine one, so R Q r has
  // zero mean already: the projection of bc removes rounding only.)
  if (!rc && p.remove_const_field) rc = mxg_mv_remove_const_field(r);
  if (!rc) { g->spmmCount++; rc = mxg_crs_apply(g->R[l], r, bc); }
  if (!rc && p.remove_const_field) rc = mxg_mv_remove_const_field(bc);
  // coarse-grid correction from a zero initial guess
  if (!rc) rc = vcycle<T>(g, l + 1, xc, bc, true);
  // x += P e (refine, :438-443); with "remove const field" the refined correction is cleaned before it is added
  if (!rc && p.remove_const_field) {
    g->spmmCount++;
    rc = mxg_crs_apply(g->P[l], xc, r);
    if (!rc) rc = mxg_mv_remove_const_field(r);
    if (!rc) rc = mxg_mv_add_mv(x, one, x, one, r);
  } else if (!rc) { g->spmmCount++; rc = mxg_crs_apply_axpby(g->P[l], one, xc, one, x); }
  if (!rc) rc = smooth<T>(g, l, x, b, p.smoother_degree, p.eig_ratio, false);
  mxg_mv_destroy(r);
  mxg_mv_destroy(bc);
  mxg_mv_destroy(xc);
  return rc;
}

// lambda_max(D^-1 A) by power iteration on one random vector
template <class T>
int estimateLambdaMax(mxg_gmg* g, int l, int iters, double* out) {
  const mxg_crs* A = g->A[l];
  mxg_ctx* ctx = g->ctx;
  mxg_mv *u = nullptr, *t = nullptr;
  int rc = mxg_mv_create(A->rowMap, 1, g->isComplex, &u);
  if (rc) return rc;
  if ((rc = mxg_mv_create(A->rowMap, 1, g->isComplex, &t))) { mxg_mv_destroy(u); return rc; }
  mxg_mv_random(u, 0x5eedull + l);
  double lam = 1.0, nrm = 0.0;
  for (int it = 0; it < iters && !rc; ++it) {
    rc = mxg_mv_norm2(u, &nrm);
    if (rc || nrm == 0.0) break;
    const double inv[2] = {1.0 / nrm, 0.0};
    mxg_mv_scale(u, inv);
    rc = mxg_crs_apply(A, u, t);
    if (rc) break;
    if (A->nRows > 0) {
      k_diag_scale<T><<<gridCols(ctx, A->nRows, 1), kBlock, 0, ctx->stream>>>(tableOf<T>(u), tableOf<T>(t), static_cast<const T*>(A->dInvDiag), A->nRows);
      LAUNCH_CHECK(ctx);
    }
    rc = mxg_mv_norm2(u, &lam);  // |D^-1 A u| with |u| = 1
  }
  mxg_mv_destroy(u);
  mxg_mv_destroy(t);
  *out = lam;
  return rc;
}

int ensureWork(mxg_gmg* g, int ncols) {
  if (g->workCols >= ncols) return MXG_OK;
  for (auto* vec : {&g->x, &g->b, &g->v, &g->w})
    for (auto& m : *vec) {
      if (m) mxg_mv_destroy(m);
      m = nullptr;
    }
  for (int l = 0; l < g->nlevels; ++l) {
    int rc;
    if ((rc = mxg_mv_create(g->A[l]->rowMap, ncols, g->isComplex, &g->x[l]))) return rc;
    if ((rc = mxg_mv_create(g->A[l]->rowMap, ncols, g->isComplex, &g->b[l]))) return rc;
    if ((rc = mxg_mv_create(g->A[l]->rowMap, ncols, g->isComplex, &g->v[l]))) return rc;
    if ((rc = mxg_mv_create(g->A[l]->rowMap, ncols, g->isComplex, &g->w[l]))) return rc;
  }
  g->workCols = ncols;
  return MXG_OK;
}

template <class T>
int applyImpl(mxg_gmg* g, const mxg_mv* b, mxg_mv* x) {
  const int nc = b->ncols;
  int rc = ensureWork(g, nc);
  if (rc) return rc;
  const mxg_gmg_params& p = g->prm;
  const double zero[2] = {0, 0};
  if (!p.full_multigrid || g->nlevels == 1) {
    rc = vcycle<T>(g, 0, x, b, true);
    for (int c = 1; c < p.cycles && !rc; ++c) rc = vcycle<T>(g, 0, x, b, false);
    return rc;
  }
  // full multigrid (MxGeoMultigridPrec.cpp:547-616): restrict b to every level, solve coarsest,
  // then interpolate up, running `cycles` V-cycles from each level
  std::vector<mxg_mv*> bl(g->nlevels, nullptr), xl(g->nlevels, nullptr);
  bl[0] = const_cast<mxg_mv*>(b);
  xl[0] = x;
  for (int l = 1; l < g->nlevels && !rc; ++l) {
    if ((rc = viewCols(g->b[l], nc, &bl[l]))) break;
    if ((rc = viewCols(g->x[l], nc, &xl[l]))) break;
    g->spmmCount++;
    rc = mxg_crs_apply(g->R[l - 1], bl[l - 1], bl[l]);
    if (!rc && p.remove_const_field) rc = mxg_mv_remove_const_field(bl[l]);
  }
  const int last = g->nlevels - 1;
  if (!rc) rc = smooth<T>(g, last, xl[last], bl[last], p.coarse_degree, p.coarse_eig_ratio, true);
  for (int l = last - 1; l >= 0 && !rc; --l) {
    g->spmmCount++;
    rc = mxg_crs_apply(g->P[l], xl[l + 1], xl[l]);
    if (!rc && p.remove_const_field) rc = mxg_mv_remove_const_field(xl[l]);
    // the coarse work vectors b[l+1], x[l+1] are reused inside vcycle(l): stash what is still needed
    // (nothing: levels below l are finished once their solution has been interpolated up)
    for (int c = 0; c < p.cycles && !rc; ++c) rc = vcycle<T>(g, l, xl[l], bl[l], false);
  }
  for (int l = 1; l < g->nlevels; ++l) {
    if (bl[l]) mxg_mv_destroy(bl[l]);
    if (xl[l]) mxg_mv_destroy(xl[l]);
  }
  (void)zero;
  return rc;
}

}  // namespace

extern "C" {

void mxg_gmg_default_params(mxg_gmg_params* p) {
  if (!p) return;
  p->smoother_degree = 2;      // "linear solver : smoother sweeps"
  p->eig_ratio = 30.0;         // ChebList "chebyshev: ratio eigenvalue" (MxGeoMultigridPrec.cpp:117-120)
  p->cycles = 1;               // "linear solver : cycles"
  p->coarse_degree = 30;
  p->coarse_eig_ratio = 1000.0;
  p->full_multigrid = 0;
  p->power_iterations = 30;
  p->remove_const_field = 0;   // "linear solver : remove const field" default (MxGeoMultigridPrec.cpp:108)
}

int mxg_gmg_create(mxg_ctx* ctx, int nlevels, mxg_crs* const* ops, mxg_crs* const* restrictors, mxg_crs* const* prolongators,
                   const mxg_gmg_params* params, mxg_gmg** out) {
  MXG_REQUIRE(ctx && ops && out && nlevels >= 1, "mxg_gmg_create: bad argument");
  MXG_REQUIRE(nlevels == 1 || (restrictors && prolongators), "mxg_gmg_create: transfer operators missing");
  MXG_REQUIRE(ops[0] != nullptr, "mxg_gmg_create: level 0 operator is NULL");
  mxg_gmg* g = new mxg_gmg;
  g->ctx = ctx;
  g->nlevels = nlevels;
  if (params) g->prm = *params; else mxg_gmg_default_params(&g->prm);
  g->isComplex = ops[0]->isComplex;
  for (int l = 0; l < nlevels; ++l) {
    const mxg_crs* A = ops[l];
    if (!A || A->ctx != ctx || A->isComplex != g->isComplex || !A->dInvDiag) {
      delete g;
      setError("mxg_gmg_create: level %d operator is missing, on another context, of another scalar type or not square", l);
      return MXG_ERR_ARG;
    }
    g->A.push_back(A);
    if (l + 1 < nlevels) {
      const mxg_crs *R = restrictors[l], *P = prolongators[l];
      if (!R || !P || R->nLoc != A->nRows || R->nRows != ops[l + 1]->nRows || P->nRows != A->nRows || P->nLoc != ops[l + 1]->nRows) {
        delete g;
        setError("mxg_gmg_create: transfer operators of level %d do not match the level sizes", l);
        return MXG_ERR_ARG;
      }
      g->R.push_back(R);
      g->P.push_back(P);
    }
  }
  g->x.assign(nlevels, nullptr);
  g->b.assign(nlevels, nullptr);
  g->v.assign(nlevels, nullptr);
  g->w.assign(nlevels, nullptr);
  g->lambdaMax.assign(nlevels, 1.0);
  MXG_CUDA(cudaSetDevice(ctx->device));
  for (int l = 0; l < nlevels; ++l) {
    int rc = g->isComplex ? estimateLambdaMax<zd>(g, l, g->prm.power_iterations, &g->lambdaMax[l])
                          : estimateLambdaMax<double>(g, l, g->prm.power_iterations, &g->lambdaMax[l]);
    if (rc) {
      mxg_gmg_destroy(g);
      return rc;
    }
  }
  *out = g;
  return MXG_OK;
}

int mxg_gmg_destroy(mxg_gmg* g) {
  if (!g) return MXG_OK;
  for (auto* vec : {&g->x, &g->b, &g->v, &g->w})
    for (auto& m : *vec)
      if (m) mxg_mv_destroy(m);
  delete g;
  return MXG_OK;
}

int mxg_gmg_apply(mxg_gmg* g, const mxg_mv* b, mxg_mv* x) {
  MXG_REQUIRE(g && b && x, "mxg_gmg_apply: NULL argument");
  MXG_REQUIRE(b->ld == g->A[0]->nRows && x->ld == g->A[0]->nRows, "mxg_gmg_apply: vector length does not match the fine level");
  MXG_REQUIRE(b->ncols == x->ncols, "mxg_gmg_apply: column counts differ");
  MXG_REQUIRE(b->isComplex == g->isComplex && x->isComplex == g->isComplex, "mxg_gmg_apply: mixed real/complex operands");
  for (void* pb : b->col)
    for (void* px : x->col) MXG_REQUIRE(pb != px, "mxg_gmg_apply: x and b must not alias");
  MXG_CUDA(cudaSetDevice(g->ctx->device));
  return g->isComplex ? applyImpl<zd>(g, b, x) : applyImpl<double>(g, b, x);
}

int mxg_gmg_info(const mxg_gmg* g, int level, double out[4]) {
  MXG_REQUIRE(g && out && level >= 0 && level < g->nlevels, "mxg_gmg_info: bad argument");
  out[0] = double(g->A[level]->nRows);
  out[1] = double(g->A[level]->nnz);
  out[2] = g->lambdaMax[level];
  out[3] = double(g->spmmCount);
  return MXG_OK;
}

// y = d .* x  (diagonal operators such as mRhs = dmA, MxMagWaveOp.cpp:865,895)
int mxg_mv_diag_mult(mxg_mv* y, const mxg_mv* d, const mxg_mv* x) {
  MXG_REQUIRE(y && d && x, "mxg_mv_diag_mult: NULL argument");
  MXG_REQUIRE(d->ncols == 1 && d->ld == x->ld && y->ld == x->ld && y->ncols == x->ncols, "mxg_mv_diag_mult: shape mismatch");
  MXG_REQUIRE(d->isComplex == x->isComplex && y->isComplex == x->isComplex, "mxg_mv_diag_mult: mixed real/complex operands");
  mxg_ctx* ctx = x->map->ctx;
  if (x->ld == 0) return MXG_OK;
  MXG_CUDA(cudaSetDevice(ctx->device));
  if (x->isComplex)
    k_diag_scale<zd><<<gridCols(ctx, x->ld, x->ncols), kBlock, 0, ctx->stream>>>(tableOf<zd>(y), tableOf<zd>(x), static_cast<const zd*>(d->col[0]), x->ld);
  else
    k_diag_scale<double><<<gridCols(ctx, x->ld, x->ncols), kBlock, 0, ctx->stream>>>(tableOf<double>(y), tableOf<double>(x), static_cast<const double*>(d->col[0]), x->ld);
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}

}  // extern "C"

// y = D^-1 x with D = diag(A): Jacobi preconditioner for the scalar-Laplacian projection solve
// (the reference uses ML/ILUT there, MxMagWaveOp.cpp:285-537)
extern "C" int mxg_crs_jacobi(const mxg_crs* A, const mxg_mv* x, mxg_mv* y) {
  MXG_REQUIRE(A && x && y, "mxg_crs_jacobi: NULL argument");
  MXG_REQUIRE(A->dInvDiag != nullptr, "mxg_crs_jacobi: operator is not square on one map");
  MXG_REQUIRE(x->ld == A->nRows && y->ld == A->nRows && x->ncols == y->ncols, "mxg_crs_jacobi: shape mismatch");
  MXG_REQUIRE(x->isComplex == A->isComplex && y->isComplex == A->isComplex, "mxg_crs_jacobi: mixed real/complex operands");
  mxg_ctx* ctx = A->ctx;
  if (x->ld == 0) return MXG_OK;
  MXG_CUDA(cudaSetDevice(ctx->device));
  if (A->isComplex)
    k_diag_scale<zd><<<gridCols(ctx, x->ld, x->ncols), kBlock, 0, ctx->stream>>>(tableOf<zd>(y), tableOf<zd>(x), static_cast<const zd*>(A->dInvDiag), x->ld);
  else
    k_diag_scale<double><<<gridCols(ctx, x->ld, x->ncols), kBlock, 0, ctx->stream>>>(tableOf<double>(y), tableOf<double>(x), static_cast<const double*>(A->dInvDiag), x->ld);
  LAUNCH_CHECK(ctx);
  return MXG_OK;
}
