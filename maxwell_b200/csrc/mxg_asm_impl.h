// Operator assembly on an executor (SURVEY 8 f2): the simulation set-up of MxEMSim (fields, boundary conditions, DOF
// maps), the named operators of MxEMOps / MxMagWaveOp::initMatrices and the CRS algebra they are chained with. The
// executor X supplies memory, a parallel for-each over rows, a prefix scan and a maximum; mxg_asm.cu instantiates this
// with CUDA kernels (the product), tests/cpp/asm_replay.cpp with plain loops (CPU replay of the same row functions).
//
// Reference: MxEMSim.cpp:54-199 (set-up order), MxYeeElecFieldBase.cpp:89-138 / MxYeeMagFieldBase.cpp:119-168 /
// MxYeePsiField.cpp:74-97 (wall translation), MxGridField.cpp:34-38 (phase factors), MxEMOps.cpp:39-168 and
// MxMagWaveOp.cpp:137-245 (operator chains), MxCrsMatrix.cpp:358-430 (multiply / add).
#pragma once
#include <cmath>
#include <complex>
#include <cstring>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <vector>

#include "mxg_yee.h"
#include "mxg_shape.h"
#include "mxg_eps.h"

namespace mxa {

using mxy::Cx;

// A CRS matrix on the executor. It stores nrows of the mapRows rows of its row field's map: from map position rowBegin
// on, except that the last run2Rows of them continue at run2Begin (a second run, which only the chains of buildOpRows
// create on periodic-x grids). Columns are always positions in the whole column map. A whole-map matrix has
// rowBegin = 0 and nrows = mapRows.
template <class S>
struct Csr {
  int64_t nrows = 0, ncols = 0, nnz = 0;
  int64_t* rowptr = nullptr;
  int32_t* col = nullptr;
  S* val = nullptr;
  int rowField = -1, colField = -1;   // which field maps the rows / columns live on
  int64_t rowBegin = 0, mapRows = 0, run2Begin = 0, run2Rows = 0;
  mxy::RowRuns runs() const { return {{rowBegin, run2Begin}, {nrows - run2Rows, run2Rows}}; }
  void setRuns(const mxy::RowRuns& r, int64_t rowsOfMap) {
    rowBegin = r.begin[0]; run2Begin = r.begin[1]; run2Rows = r.count[1]; mapRows = rowsOfMap;
  }
  bool partial() const { return rowBegin != 0 || nrows != mapRows; }
  mxy::CsrView<S> view() const { return {nrows, ncols, rowptr, col, val, runs()}; }
};

// every map position of `inner` is stored in `outer`
inline bool covers(const mxy::RowRuns& outer, const mxy::RowRuns& inner) {
  for (int r = 0; r < 2; ++r) {
    int64_t k = inner.begin[r];
    const int64_t end = inner.begin[r] + inner.count[r];
    while (k < end) {
      int64_t next = -1;
      for (int o = 0; o < 2; ++o)
        if (k >= outer.begin[o] && k < outer.begin[o] + outer.count[o]) next = outer.begin[o] + outer.count[o];
      if (next < 0) return false;
      k = next;
    }
  }
  return true;
}
inline bool sameRuns(const mxy::RowRuns& a, const mxy::RowRuns& b) {
  for (int r = 0; r < 2; ++r)
    if (a.count[r] != b.count[r] || (a.count[r] > 0 && a.begin[r] != b.begin[r])) return false;
  return true;
}

template <class S> inline S scalarFrom(double re, double im);
template <> inline double scalarFrom<double>(double re, double) { return re; }
template <> inline Cx scalarFrom<Cx>(double re, double im) { return {re, im}; }

template <class S>
struct ScaleVals {
  S* val;
  S s;
  MXY_HD void operator()(int64_t i) const { val[i] = mxy::mulS(val[i], s); }
};
struct RowLen2 {      // |row i of A| + |row i of B|
  const int64_t *a, *b;
  MXY_HD int operator()(int64_t i) const { return int((a[i + 1] - a[i]) + (b ? b[i + 1] - b[i] : 0)); }
};
template <class Fn>
struct StoreInt {
  Fn fn;
  int32_t* out;
  MXY_HD void operator()(int64_t i) const { out[i] = fn(i); }
};

// executor memory released at scope exit (temporaries of the passes below; an exception must not leak them)
template <class X, class T>
struct Scoped {
  X& x;
  T* p;
  Scoped(X& exec, int64_t n) : x(exec), p(exec.template alloc<T>(n)) {}
  ~Scoped() { x.free(p); }
  Scoped(const Scoped&) = delete;
  Scoped& operator=(const Scoped&) = delete;
  T* release() { T* q = p; p = nullptr; return q; }
};

// one factor of an operator chain: a generator (op = mxy::GenOp with its fraction arguments), the simulation's
// dielectric rows (kEps, kEpsVolAve), or a matrix handed in for the latter (given)
constexpr int kEps = 100, kEpsVolAve = 101;
template <class S>
struct Factor {
  int op;
  int fracField = 0;
  bool inverse = false;
  double minFrac = 0.0;
  const Csr<S>* given = nullptr;
};

template <class X>
class Assembler {
 public:
  static constexpr int kGenRowField[4] = {mxy::FIELD_B, mxy::FIELD_E, mxy::FIELD_PSI, mxy::FIELD_B};
  static constexpr int kGenColField[4] = {mxy::FIELD_E, mxy::FIELD_B, mxy::FIELD_B, mxy::FIELD_PSI};
  explicit Assembler(X& x) : x_(x) { std::memset(&h_, 0, sizeof(h_)); }
  ~Assembler() {
    for (int k = 0; k < mxy::NUM_FIELDS; ++k) {
      x_.free(const_cast<double*>(h_.f[k].region));
      x_.free(const_cast<int32_t*>(h_.f[k].lidOf));
      x_.free(const_cast<int64_t*>(h_.f[k].gids));
    }
    x_.free(const_cast<double*>(h_.f[mxy::FIELD_D].region));      // D borrows E's map
    for (int d = 0; d < h_.numDiel; ++d) {
      x_.free(const_cast<double*>(h_.diel[d].fracE));
      x_.free(const_cast<double*>(h_.diel[d].fracD));
      x_.free(const_cast<double*>(h_.diel[d].fracPsi));
      x_.free(const_cast<void*>(h_.diel[d].shape));
    }
    x_.free(h_.err);
    x_.free(dSim_);
  }
  Assembler(const Assembler&) = delete;
  Assembler& operator=(const Assembler&) = delete;

  X& exec() { return x_; }
  const mxy::Sim& sim() const { return h_; }
  bool hasPEC() const { return hasPEC_; }
  bool isSetUp() const { return setUp_; }

  // MxEMSim.cpp:54-120: grid, the three Yee fields, wall translation, Bloch phases
  void init(const int n[3], const double origin[3], const double size[3], const int lower[3], const int upper[3],
            const double phaseShifts[3], double dmFrac, int literalUpperPeriodicE) {
    for (int i = 0; i < 3; ++i) {
      if (n[i] < 1) throw std::runtime_error("grid needs at least one cell per direction");
      h_.g.N[i] = n[i];
      h_.g.origin[i] = origin[i];
      h_.g.d[i] = size[i] / double(n[i]);
    }
    if (mxy::numNodes(h_.g) * 3 >= (int64_t(1) << 31)) throw std::runtime_error("grid too large for 32-bit DOF ids");
    const double dx = h_.g.d[0], dy = h_.g.d[1], dz = h_.g.d[2];
    std::complex<double> phase[3];
    for (int i = 0; i < 3; ++i) phase[i] = std::exp(std::complex<double>(0.0, 1.0) * phaseShifts[i]);   // MxGridField.cpp:34-38
    complex_ = phaseShifts[0] != 0 || phaseShifts[1] != 0 || phaseShifts[2] != 0;
    for (int i = 0; i < 3; ++i) phase_[i] = phaseShifts[i];
    for (int k = 0; k < mxy::NUM_ALL_FIELDS; ++k) {
      mxy::Field& f = h_.f[k];
      f.kind = k;
      f.ncomp = k == mxy::FIELD_PSI ? 1 : 3;
      for (auto& r : f.xi) for (double& v : r) v = 0.0;
      if (k == mxy::FIELD_E || k == mxy::FIELD_D) {  // MxYeeElecFieldBase.cpp:64-82 (D: same positions, MxYeeFitDField)
        f.xi[0][0] = 0.5 * dx; f.xi[1][1] = 0.5 * dy; f.xi[2][2] = 0.5 * dz;
      } else if (k == mxy::FIELD_B) {                // MxYeeMagFieldBase.cpp:85-116
        f.xi[0][1] = 0.5 * dy; f.xi[0][2] = 0.5 * dz;
        f.xi[1][2] = 0.5 * dz; f.xi[1][0] = 0.5 * dx;
        f.xi[2][0] = 0.5 * dx; f.xi[2][1] = 0.5 * dy;
      } else {                                       // MxYeePsiField.cpp:51-72
        f.xi[0][0] = 0.5 * dx; f.xi[0][1] = 0.5 * dy; f.xi[0][2] = 0.5 * dz;
      }
      for (int c = 0; c < 3; ++c)
        for (int i = 0; i < 3; ++i) {
          f.lbc[c][i] = translateBC(k, lower[i], c, i);
          f.ubc[c][i] = translateBC(k, upper[i], c, i);
        }
      f.dmFrac = k == mxy::FIELD_B ? dmFrac : 0.0;
      f.regionSet = 0;
      f.literalUpperPeriodicE = literalUpperPeriodicE;
      for (int code = 0; code < 125; ++code) {       // MxGridField.cpp:145-190, direction 0 first
        const int act[3] = {code / 25, (code / 5) % 5, code % 5};
        std::complex<double> res(1.0, 0.0);
        for (int i = 0; i < 3; ++i) {
          if (act[i] == mxy::ACT_DIV) res /= phase[i];
          else if (act[i] == mxy::ACT_MUL) res *= phase[i];
          else if (act[i] == mxy::ACT_NEG) res *= -1.0;
          else if (act[i] == mxy::ACT_ZERO) res *= 0.0;
        }
        f.facRe[code] = res.real();
        f.facIm[code] = res.imag();
      }
    }
    h_.err = x_.template alloc<int>(1);
    const int zero = 0;
    x_.toExec(h_.err, &zero, sizeof(int));
    dSim_ = x_.template alloc<mxy::Sim>(1);
    pushSim();
  }

  // PEC fractions of one field on the guarded block ((N+3)^3 cells x ncomp), host array as MxGridField keeps it
  // (MxGridField.hpp:259-279). All three fields must be given before setup() when a PEC shape exists.
  void setRegionFromHost(int kind, const double* fracs) {
    mxy::Field& f = h_.f[kind];
    const int64_t n = mxy::numFullCells(h_.g) * f.ncomp;
    double* d = regionBuffer(kind);
    x_.toExec(d, fracs, size_t(n) * sizeof(double));
    pushSim();
  }
  // the executor-side fraction array of a field (filled by the fraction kernels)
  double* regionBuffer(int kind) {
    mxy::Field& f = h_.f[kind];
    if (!f.region) f.region = x_.template alloc<double>(mxy::numFullCells(h_.g) * f.ncomp);
    f.regionSet = 1;
    hasPEC_ = true;
    setUp_ = false;
    return const_cast<double*>(f.region);
  }
  void regionChanged() { pushSim(); }

  // PEC region from a shape: edge / face / cell fractions of B, E and psi computed on the executor
  // (MxEMSim.cpp:122-129 -> MxGridField::addShapeRep, MxGridField.cpp:193-226)
  void setPecShape(const Shape& shape) {
    checkShape(shape);
    ShapeNode* nodes = uploadShape(shape);
    for (int k = 0; k < mxy::NUM_FIELDS; ++k) {
      double* out = regionBuffer(k);
      pushSim();
      x_.forEach(mxy::numFullCells(h_.g), FractionCells{dSim_, nodes, k, out});
    }
    x_.sync();
    x_.free(nodes);
    pec_ = shape;
    // fractions of the dual faces are only needed next to dielectrics; drop stale ones
    x_.free(const_cast<double*>(h_.f[mxy::FIELD_D].region));
    h_.f[mxy::FIELD_D].region = nullptr;
    pushSim();
  }

  // MxEMSim::addDielectric + MxEMSim.cpp:134-148: fractions of the dielectric's shape on E, D and psi; eps = 3x3 complex
  // tensor, row-major (re, im) pairs
  void addDielectric(const Shape& shape, const double eps[18]) {
    checkShape(shape);
    if (h_.numDiel >= mxy::kMaxDielectrics) throw std::runtime_error("at most 4 dielectric objects");
    mxy::DielectricRep& D = h_.diel[h_.numDiel];
    ShapeNode* nodes = uploadShape(shape);
    const int64_t cells = mxy::numFullCells(h_.g);
    double* fe = x_.template alloc<double>(cells * 3);
    double* fd = x_.template alloc<double>(cells * 3);
    double* fp = x_.template alloc<double>(cells);
    x_.forEach(cells, FractionCells{dSim_, nodes, mxy::FIELD_E, fe});
    x_.forEach(cells, FractionCells{dSim_, nodes, mxy::FIELD_D, fd});
    x_.forEach(cells, FractionCells{dSim_, nodes, mxy::FIELD_PSI, fp});
    x_.sync();
    D.fracE = fe; D.fracD = fd; D.fracPsi = fp;
    D.shape = nodes;
    bool offDiag = false;
    for (int i = 0; i < 9; ++i) { D.epsRe[i] = eps[2 * i]; D.epsIm[i] = eps[2 * i + 1]; }
    for (int i : {1, 2, 5}) offDiag = offDiag || D.epsRe[i] != 0.0 || D.epsIm[i] != 0.0;    // MxDielectric.cpp:27-36
    D.isDiag = offDiag ? 0 : 1;
    h_.numDiel++;
    pushSim();
  }
  int numDielectrics() const { return h_.numDiel; }

  // MxGridField.cpp:256-297 for B, E and psi (B first: the others consult its rules)
  void setup() {
    if (hasPEC_)
      for (int k = 0; k < mxy::NUM_FIELDS; ++k)
        if (!h_.f[k].region) throw std::runtime_error("a PEC region needs fractions for the B, E and psi fields");
    if (hasPEC_ && h_.numDiel > 0 && !h_.f[mxy::FIELD_D].region) {     // MxEMSim.cpp:122-129: the D field joins with dielectrics
      if (pec_.nodes.empty()) throw std::runtime_error("dielectrics next to host-supplied PEC fractions need those of the D field too (dfield)");
      ShapeNode* nodes = uploadShape(pec_);
      double* out = x_.template alloc<double>(mxy::numFullCells(h_.g) * 3);
      x_.forEach(mxy::numFullCells(h_.g), FractionCells{dSim_, nodes, mxy::FIELD_D, out});
      x_.sync();
      x_.free(nodes);
      h_.f[mxy::FIELD_D].region = out;
    }
    h_.f[mxy::FIELD_D].regionSet = hasPEC_ ? 1 : 0;
    for (int k = 0; k < mxy::NUM_FIELDS; ++k) {
      mxy::Field& f = h_.f[k];
      x_.free(const_cast<int32_t*>(f.lidOf));
      x_.free(const_cast<int64_t*>(f.gids));
      f.lidOf = nullptr; f.gids = nullptr; f.nLoc = 0;
      const int64_t n = mxy::numNodes(h_.g) * f.ncomp;
      Scoped<X, int32_t> flag(x_, n);
      Scoped<X, int64_t> off(x_, n + 1);
      x_.forEach(n, mxy::MapFlags{dSim_, k, flag.p});
      const int64_t total = x_.scan(flag.p, off.p, n);
      Scoped<X, int32_t> lid(x_, n);
      Scoped<X, int64_t> gids(x_, total > 0 ? total : 1);
      x_.forEach(n, mxy::MapFill{flag.p, off.p, lid.p, gids.p});
      x_.sync();
      f.lidOf = lid.release();
      f.gids = gids.release();
      f.nLoc = total;
      pushSim();
      // first map position of every x-plane: the row runs of slab-partitioned chains
      const int64_t np = h_.g.N[0] + 2;
      Scoped<X, int64_t> ps(x_, np);
      x_.forEach(np, mxy::PlaneStart{f.gids, total, planeGids(k), ps.p});
      planeStart_[k].assign(size_t(np), 0);
      x_.toHost(planeStart_[k].data(), ps.p, size_t(np) * sizeof(int64_t));
    }
    h_.f[mxy::FIELD_D].lidOf = h_.f[mxy::FIELD_E].lidOf;      // MxEMSim.cpp:186-190: D shares E's map
    h_.f[mxy::FIELD_D].gids = h_.f[mxy::FIELD_E].gids;
    h_.f[mxy::FIELD_D].nLoc = h_.f[mxy::FIELD_E].nLoc;
    pushSim();
    checkErr("map set-up");
    setUp_ = true;
  }

  int64_t mapSize(int kind) const { return h_.f[kind].nLoc; }
  int64_t numGlobal(int kind) const { return mxy::numNodes(h_.g) * h_.f[kind].ncomp; }
  void copyMap(int kind, int64_t* out) { x_.toHost(out, h_.f[kind].gids, size_t(h_.f[kind].nLoc) * sizeof(int64_t)); }
  const int64_t* mapGids(int kind) const { return h_.f[kind].gids; }   // executor memory, mapSize(kind) ascending GIDs
  void copyFractions(int kind, double* out) {
    const mxy::Field& f = h_.f[kind];
    if (!f.region) throw std::runtime_error("field has no PEC fractions");
    x_.toHost(out, f.region, size_t(mxy::numFullCells(h_.g) * f.ncomp) * sizeof(double));
  }

  // ---- CRS algebra ------------------------------------------------------------------------------------------
  template <class S>
  void destroy(Csr<S>& m) {
    x_.free(m.rowptr); x_.free(m.col); x_.free(m.val);
    m = Csr<S>();
  }

  template <class S, class RowFn>
  Csr<S> buildRows(int64_t nrows, int64_t ncols, const RowFn& fn) {
    Csr<S> m;
    m.nrows = nrows; m.ncols = ncols; m.mapRows = nrows;
    Scoped<X, int64_t> rowptr(x_, nrows + 1);
    {
      Scoped<X, int32_t> cnt(x_, nrows > 0 ? nrows : 1);
      x_.forEach(nrows, mxy::CountRows<S, RowFn>{fn, cnt.p});
      m.nnz = x_.scan(cnt.p, rowptr.p, nrows);
    }
    Scoped<X, int32_t> col(x_, m.nnz > 0 ? m.nnz : 1);
    Scoped<X, S> val(x_, m.nnz > 0 ? m.nnz : 1);
    x_.forEach(nrows, mxy::FillRows<S, RowFn>{fn, rowptr.p, col.p, val.p});
    m.rowptr = rowptr.release();
    m.col = col.release();
    m.val = val.release();
    return m;
  }

  template <class Fn>
  int maxOverRows(int64_t nrows, const Fn& fn) {
    if (nrows == 0) return 0;
    Scoped<X, int32_t> tmp(x_, nrows);
    x_.forEach(nrows, StoreInt<Fn>{fn, tmp.p});
    return x_.maxOf(tmp.p, nrows);
  }

  // Rows of A * B on A's stored rows. B may store only some of its rows: the rows A's columns reference.
  template <class S>
  Csr<S> multiply(const Csr<S>& A, const Csr<S>& B) {       // MxCrsMatrix.cpp:358-382
    if (A.ncols != B.mapRows) throw std::runtime_error("multiply: shapes do not match");
    if (B.partial() && maxOverRows(A.nrows, mxy::MissingCols<S>{A.view(), B.runs()}) > 0)
      throw std::runtime_error("multiply: a column of A has no stored row in B");
    const mxy::CsrView<S> a = A.view(), b = B.view();
    const int bound = maxOverRows(A.nrows, mxy::ProductBound<S>{a, b, h_.err});
    Csr<S> C;
    if (bound <= 16) C = buildRows<S>(A.nrows, B.ncols, mxy::ProductRow<S, 16>{a, b, h_.err});
    else if (bound <= 32) C = buildRows<S>(A.nrows, B.ncols, mxy::ProductRow<S, 32>{a, b, h_.err});
    else if (bound <= 64) C = buildRows<S>(A.nrows, B.ncols, mxy::ProductRow<S, 64>{a, b, h_.err});
    else if (bound <= 160) C = buildRows<S>(A.nrows, B.ncols, mxy::ProductRow<S, 160>{a, b, h_.err});
    else if (bound <= 400) C = buildRows<S>(A.nrows, B.ncols, mxy::ProductRow<S, 400>{a, b, h_.err});
    else throw std::runtime_error("multiply: a product row would exceed 400 entries");
    C.setRuns(A.runs(), A.mapRows);
    C.rowField = A.rowField;
    C.colField = B.colField;
    struct Release {
      Assembler* as; Csr<S>* c; bool keep = false;
      ~Release() { if (!keep) as->destroy(*c); }
    } guard{this, &C};
    checkErr("multiply");
    guard.keep = true;
    return C;
  }

  // sa A + sb B on A's stored rows; B must store them too
  template <class S>
  Csr<S> add(const Csr<S>& A, S sa, const Csr<S>& Bin, S sb, bool purge) {   // MxCrsMatrix.cpp:401-430 (+ :84-117)
    if (A.mapRows != Bin.mapRows || A.ncols != Bin.ncols) throw std::runtime_error("add: shapes do not match");
    Csr<S> sel;
    struct Owned {
      Assembler* a; Csr<S>* x;
      ~Owned() { a->destroy(*x); }
    } owned{this, &sel};
    if (!sameRuns(A.runs(), Bin.runs())) sel = selectRows(Bin, A.runs());
    const Csr<S>& B = sel.rowptr ? sel : Bin;
    const int bound = maxOverRows(A.nrows, RowLen2{A.rowptr, B.rowptr});
    Csr<S> C;
    const int p = purge ? 1 : 0;
    if (bound <= 32) C = buildRows<S>(A.nrows, A.ncols, mxy::SumRow<S, 32>{A.view(), B.view(), sa, sb, p});
    else if (bound <= 160) C = buildRows<S>(A.nrows, A.ncols, mxy::SumRow<S, 160>{A.view(), B.view(), sa, sb, p});
    else if (bound <= 800) C = buildRows<S>(A.nrows, A.ncols, mxy::SumRow<S, 800>{A.view(), B.view(), sa, sb, p});
    else throw std::runtime_error("add: a row would exceed 800 entries");
    C.setRuns(A.runs(), A.mapRows);
    C.rowField = A.rowField;
    C.colField = A.colField;
    return C;
  }

  // a copy of the map rows `over` of A
  template <class S>
  Csr<S> selectRows(const Csr<S>& A, const mxy::RowRuns& over) {
    if (!covers(A.runs(), over)) throw std::runtime_error("a factor does not store the rows the product needs (a column of A has no stored row in B)");
    Csr<S> m;
    m.nrows = over.size(); m.ncols = A.ncols;
    Scoped<X, int64_t> rowptr(x_, m.nrows + 1);
    {
      Scoped<X, int32_t> cnt(x_, m.nrows > 0 ? m.nrows : 1);
      x_.forEach(m.nrows, mxy::SelectCount<S>{A.view(), over, cnt.p});
      m.nnz = x_.scan(cnt.p, rowptr.p, m.nrows);
    }
    Scoped<X, int32_t> col(x_, m.nnz > 0 ? m.nnz : 1);
    Scoped<X, S> val(x_, m.nnz > 0 ? m.nnz : 1);
    x_.forEach(m.nrows, mxy::SelectFill<S>{A.view(), over, rowptr.p, col.p, val.p});
    x_.sync();
    m.rowptr = rowptr.release();
    m.col = col.release();
    m.val = val.release();
    m.setRuns(over, A.mapRows);
    m.rowField = A.rowField;
    m.colField = A.colField;
    return m;
  }

  template <class S>
  Csr<S> purgeZeros(const Csr<S>& A) {                      // MxCrsMatrix.cpp:84-117
    const int bound = maxOverRows(A.nrows, RowLen2{A.rowptr, nullptr});
    Csr<S> C;
    if (bound <= 32) C = buildRows<S>(A.nrows, A.ncols, mxy::PurgeRow<S, 32>{A.view()});
    else if (bound <= 400) C = buildRows<S>(A.nrows, A.ncols, mxy::PurgeRow<S, 400>{A.view()});
    else throw std::runtime_error("purge: a row exceeds 400 entries");
    C.setRuns(A.runs(), A.mapRows);
    C.rowField = A.rowField;
    C.colField = A.colField;
    return C;
  }

  template <class S>
  void scale(Csr<S>& A, S s) { x_.forEach(A.nnz, ScaleVals<S>{A.val, s}); }

  // host CSR (local column indices) -> executor; used for operators that are still generated on the host
  // (the dielectric invEps of MxYeeFitInvEps) so that the chains around them run here
  template <class S>
  Csr<S> upload(int64_t nrows, int64_t ncols, const int64_t* rowptr, const int32_t* col, const S* val, int rowField, int colField) {
    Csr<S> m;
    m.nrows = nrows; m.ncols = ncols; m.nnz = rowptr[nrows]; m.mapRows = nrows;
    m.rowField = rowField; m.colField = colField;
    m.rowptr = x_.template alloc<int64_t>(nrows + 1);
    m.col = x_.template alloc<int32_t>(m.nnz > 0 ? m.nnz : 1);
    m.val = x_.template alloc<S>(m.nnz > 0 ? m.nnz : 1);
    x_.toExec(m.rowptr, rowptr, size_t(nrows + 1) * sizeof(int64_t));
    x_.toExec(m.col, col, size_t(m.nnz) * sizeof(int32_t));
    x_.toExec(m.val, val, size_t(m.nnz) * sizeof(S));
    return m;
  }

  // (conjugate) transpose, rows sorted by column
  template <class S>
  Csr<S> transpose(const Csr<S>& A) {
    if (A.partial())
      throw std::runtime_error("transpose: the operand stores only some of its rows, so no column of the transpose is complete "
                               "(the rows of a restriction come from interpolator_transpose_rows)");
    return transposeWindow(A, 0, A.ncols);
  }

  // rows [c0, c1) of the (conjugate) transpose: the entries of A in the columns [c0, c1), rows sorted by column
  template <class S>
  Csr<S> transposeWindow(const Csr<S>& A, int64_t c0, int64_t c1) {
    Csr<S> T;
    T.nrows = c1 - c0; T.ncols = A.mapRows;
    T.rowBegin = c0; T.mapRows = A.ncols;
    T.rowField = A.colField; T.colField = A.rowField;
    const int32_t w0 = int32_t(c0), w1 = int32_t(c1);
    Scoped<X, int32_t> cnt(x_, T.nrows > 0 ? T.nrows : 1);
    Scoped<X, int64_t> rowptr(x_, T.nrows + 1);
    x_.zero(cnt.p, size_t(T.nrows) * sizeof(int32_t));
    x_.forEach(A.nnz, mxy::TransposeCount{A.col, w0, w1, cnt.p});
    T.nnz = x_.scan(cnt.p, rowptr.p, T.nrows);
    Scoped<X, int32_t> col(x_, T.nnz > 0 ? T.nnz : 1);
    Scoped<X, S> val(x_, T.nnz > 0 ? T.nnz : 1);
    x_.zero(cnt.p, size_t(T.nrows) * sizeof(int32_t));
    x_.forEach(A.nrows, mxy::TransposeFill<S>{A.view(), w0, w1, rowptr.p, cnt.p, col.p, val.p});
    x_.forEach(T.nrows, mxy::SortRowInPlace<S>{rowptr.p, col.p, val.p});
    x_.sync();                       // cnt is released on return
    T.rowptr = rowptr.release();
    T.col = col.release();
    T.val = val.release();
    return T;
  }

  // MxGridFieldInterpolator.cpp:28-122: `field` of the simulation `from` interpolated at the DOFs of this simulation
  // (rows: this simulation's map, columns: from's map). Both live on the same executor.
  // bloch: stencil cells that wrap across a periodic face carry the Bloch factor (mxy::InterpRow; DESIGN.md GMG-bloch).
  template <class S>
  Csr<S> interpolatorFrom(Assembler& from, int field, bool bloch = false) {
    requireSetUp();
    return interpolatorRows<S>(from, field, mxy::oneRun(0, h_.f[field].nLoc), bloch);
  }
  // ... on the rows `rows` of this simulation's map
  template <class S>
  Csr<S> interpolatorRows(Assembler& from, int field, const mxy::RowRuns& rows, bool bloch = false) {
    requireSetUp();
    from.requireSetUp();
    if (bloch) checkBlochTransfer(from, std::is_same<S, double>::value);
    using Fn = mxy::AtRows<mxy::InterpRow<S>>;
    Csr<S> m = buildRows<S>(rows.size(), from.h_.f[field].nLoc, Fn{mxy::InterpRow<S>{from.dSim_, dSim_, field, bloch ? 1 : 0}, rows});
    m.setRuns(rows, h_.f[field].nLoc);
    m.rowField = field;
    m.colField = field;
    return m;
  }

  // Rows [c0, c1) of the restriction P^H (P = interpolatorFrom(from, field)) on from's map, without the rest of P: P is
  // generated on the fine rows whose 2x2x2 stencil can reach the coarse x-planes of [c0, c1), plus one margin plane on
  // each side, and only its entries in the columns [c0, c1) are transposed. The margin planes must contribute nothing
  // to the window; if they do, the derivation of the fine rows was wrong and the rows would be short.
  template <class S>
  Csr<S> interpolatorTransposeRows(Assembler& from, int field, int64_t c0, int64_t c1, bool bloch = false) {
    requireSetUp();
    from.requireSetUp();
    if (bloch) checkBlochTransfer(from, std::is_same<S, double>::value);
    const mxy::Grid& gf = h_.g;
    const mxy::Grid& gc = from.h_.g;
    const mxy::Field& ff = h_.f[field];
    const mxy::Field& fc = from.h_.f[field];
    const int P = gf.N[0] + 1;
    std::vector<char> flag(size_t(P), 0);
    if (c1 > c0) {
      int64_t g[2];
      x_.toHost(&g[0], fc.gids + c0, sizeof(int64_t));
      x_.toHost(&g[1], fc.gids + c1 - 1, sizeof(int64_t));
      const int64_t qa = g[0] / from.planeGids(field), qb = g[1] / from.planeGids(field);
      for (int pf = 0; pf < P; ++pf)                   // InterpRow's coarse cells, x direction, for every component
        for (int comp = 0; comp < ff.ncomp && !flag[size_t(pf)]; ++comp) {
          const double point = (gf.origin[0] + double(pf) * gf.d[0]) + ff.xi[comp][0];
          const int lo = int(mxy::floorD((point - fc.xi[comp][0] - gc.origin[0]) / gc.d[0]));
          for (int a = 0; a < 2; ++a) {
            const int cell[3] = {lo + a, 0, 0};
            if (cell[0] < -1 || cell[0] > gc.N[0] + 1) continue;
            int nc[3];
            mxy::interior(gc, fc, comp, cell, nc);
            if (nc[0] >= qa && nc[0] <= qb) flag[size_t(pf)] = 1;
          }
        }
    }
    int first = 0, len = 0;
    cyclicRun(flag, first, len);
    int margin[2] = {-1, -1};
    if (len > 0 && len + 2 < P) {
      first = (first - 1 + P) % P;
      margin[0] = first;
      margin[1] = (first + len + 1) % P;
      len += 2;
    } else if (len > 0) {
      first = 0; len = P;
    }
    Csr<S> p = interpolatorRows<S>(from, field, planeRows(field, first, len), bloch);
    struct Owned {
      Assembler* a; Csr<S>* x;
      ~Owned() { a->destroy(*x); }
    } owned{this, &p};
    for (int m : margin) {
      if (m < 0) continue;
      const int64_t b = planeStart_[field][size_t(m)], n = planeStart_[field][size_t(m) + 1] - b;
      if (n == 0) continue;
      const int64_t s = p.runs().find(b);
      if (maxOverRows(n, mxy::WindowHits<S>{p.view(), s, int32_t(c0), int32_t(c1)}) > 0)
        throw std::runtime_error("interpolator_transpose_rows: a margin plane of the fine rows reaches the coarse rows; the restriction rows would be short");
    }
    Csr<S> t = transposeWindow(p, c0, c1);
    return t;
  }

  // ---- generators and chains ---------------------------------------------------------------------------------
  // GIDs per x-plane of a field (GIDs are x-major: a plane is one run of the field's map)
  int64_t planeGids(int kind) const { return int64_t(h_.f[kind].ncomp) * (h_.g.N[1] + 1) * (h_.g.N[2] + 1); }
  int64_t rowsOf(int kind) const { return h_.f[kind].nLoc; }

  // the map rows of the cyclic run of `len` x-planes from plane `first` (wrapping past the last plane): at most two runs,
  // the lower one stored first
  mxy::RowRuns planeRows(int kind, int first, int len) const {
    const std::vector<int64_t>& ps = planeStart_[kind];
    const int P = h_.g.N[0] + 1;
    if (len <= 0) return mxy::oneRun(0, 0);
    if (len >= P) return mxy::oneRun(0, h_.f[kind].nLoc);
    const int last = first + len - 1;
    if (last < P) return mxy::oneRun(ps[size_t(first)], ps[size_t(last) + 1] - ps[size_t(first)]);
    const int64_t lowEnd = ps[size_t(last - P) + 1];
    return {{0, ps[size_t(first)]}, {lowEnd, h_.f[kind].nLoc - ps[size_t(first)]}};
  }
  // the shortest cyclic run of planes holding every flagged plane: the complement of the longest cyclic gap
  static void cyclicRun(const std::vector<char>& flag, int& first, int& len) {
    const int P = int(flag.size());
    int flagged = 0;
    for (char f : flag) flagged += f ? 1 : 0;
    first = 0;
    len = flagged == 0 ? 0 : P;
    if (flagged == 0 || flagged == P) return;
    int bestStart = 0, bestLen = 0, runStart = 0, runLen = 0;
    for (int i = 0; i < 2 * P; ++i) {
      if (flag[size_t(i % P)]) { runLen = 0; continue; }
      if (runLen == 0) runStart = i;
      if (++runLen > bestLen && runLen <= P) { bestLen = runLen; bestStart = runStart; }
    }
    first = (bestStart + bestLen) % P;
    len = P - bestLen;
  }
  // The rows of the next factor that the map rows `over` of A reference: the x-planes their columns touch, as a cyclic run
  // of planes of the column field (periodic x: rank 0's rows reach the top planes), turned into map rows.
  template <class S>
  mxy::RowRuns reach(const Csr<S>& A, const mxy::RowRuns& over, int colField) {
    const int P = h_.g.N[0] + 1;
    Scoped<X, int32_t> flags(x_, P);
    x_.zero(flags.p, size_t(P) * sizeof(int32_t));
    x_.forEach(over.size(), mxy::PlaneFlags<S>{A.view(), over, h_.f[colField].gids, planeGids(colField), flags.p});
    std::vector<int32_t> h(size_t(P), 0);
    x_.toHost(h.data(), flags.p, size_t(P) * sizeof(int32_t));
    std::vector<char> flag(size_t(P), 0);
    for (int p = 0; p < P; ++p) flag[size_t(p)] = h[size_t(p)] ? 1 : 0;
    int first = 0, len = 0;
    cyclicRun(flag, first, len);
    return planeRows(colField, first, len);
  }

  template <class S>
  Csr<S> generate(int op, int fracField = 0, bool inverse = false, double minFrac = 0.0) {
    const int rf = op == mxy::GEN_FRACS ? fracField : kGenRowField[op];
    return generateRows<S>(op, fracField, inverse, minFrac, mxy::oneRun(0, h_.f[rf].nLoc));
  }
  // the map rows `rows` of a generated operator
  template <class S>
  Csr<S> generateRows(int op, int fracField, bool inverse, double minFrac, const mxy::RowRuns& rows) {
    requireSetUp();
    const int rf = op == mxy::GEN_FRACS ? fracField : kGenRowField[op];
    const int cf = op == mxy::GEN_FRACS ? fracField : kGenColField[op];
    using Fn = mxy::AtRows<mxy::GenRow<S>>;
    Csr<S> m = buildRows<S>(rows.size(), h_.f[cf].nLoc, Fn{mxy::GenRow<S>{dSim_, op, fracField, inverse ? 1 : 0, minFrac}, rows});
    m.setRuns(rows, h_.f[rf].nLoc);
    m.rowField = rf;
    m.colField = cf;
    checkErr("operator generation");
    return m;
  }

  // the row field of a named operator (-1: unknown name)
  static int opRowField(const std::string& name) {
    using namespace mxy;
    for (const char* n : {"curlE", "gradPsi", "dmA", "mRhs", "curlCurl", "gradDiv", "vecLapl"}) if (name == n) return FIELD_B;
    for (const char* n : {"curlB", "dmL", "invEps"}) if (name == n) return FIELD_E;
    for (const char* n : {"divB", "dmVInv", "invEpsVolAve", "scaLapl"}) if (name == n) return FIELD_PSI;
    return -1;
  }

  // MxEMOps.cpp:39-168 and MxMagWaveOp.cpp:137-245, the whole map. invEps / invEpsVolAve (dielectrics) are optional
  // factors handed in by the caller.
  template <class S>
  Csr<S> buildOp(const std::string& name, const Csr<S>* invEps = nullptr, const Csr<S>* invEpsVolAve = nullptr) {
    requireSetUp();
    const int rf = opRowField(name);
    if (rf < 0) throw std::runtime_error("unknown operator '" + name + "'");
    return buildOpRows<S>(name, 0, h_.f[rf].nLoc, invEps, invEpsVolAve);
  }

  // The rows [r0, r1) of a named operator, bit for bit the rows of buildOp. A chain F0 F1 ... Fk is built in two passes:
  // from left to right each factor is generated on the rows the factor to its left references (F0 on [r0, r1)), then
  // the products run from right to left, F0 (F1 (... Fk)), the association order of the reference. Handed-in dielectric
  // factors (whole or partial) must store the rows their place in the chain needs.
  template <class S>
  Csr<S> buildOpRows(const std::string& name, int64_t r0, int64_t r1, const Csr<S>* invEps = nullptr,
                     const Csr<S>* invEpsVolAve = nullptr) {
    using namespace mxy;
    requireSetUp();
    const int rf = opRowField(name);
    if (rf < 0) throw std::runtime_error("unknown operator '" + name + "'");
    if (r0 < 0 || r1 < r0 || r1 > h_.f[rf].nLoc) throw std::runtime_error("operator rows: the range is outside the row map");
    if ((name == "invEps" || name == "invEpsVolAve") && h_.numDiel == 0) throw std::runtime_error("the simulation has no dielectric objects");
    if (name == "vecLapl") {                                                       // MxMagWaveOp.cpp:183-205
      Csr<S> cc = buildOpRows<S>("curlCurl", r0, r1, invEps, invEpsVolAve);
      Csr<S> gd;
      struct Owned {
        Assembler* a; Csr<S>*x, *y;
        ~Owned() { a->destroy(*x); a->destroy(*y); }
      } owned{this, &cc, &gd};
      gd = buildOpRows<S>("gradDiv", r0, r1, invEps, invEpsVolAve);
      return add(cc, scalarFrom<S>(1.0, 0.0), gd, scalarFrom<S>(-1.0, 0.0), true);
    }
    const bool pec = hasPEC_, withEps = invEps || h_.numDiel > 0, withVol = invEpsVolAve || h_.numDiel > 0;
    // a factor: a generator (op >= 0), the dielectric rows (op = kEps / kEpsVolAve), or a handed-in matrix
    std::vector<Factor<S>> chain;
    const Factor<S> curlE{GEN_CURL_E}, curlB{GEN_CURL_B}, divB{GEN_DIV_B}, gradPsi{GEN_GRAD_PSI};
    const Factor<S> dmA{GEN_FRACS, FIELD_B, false, 0.e-12}, dmL{GEN_FRACS, FIELD_E, false, 0.e-6};     // MxEMOps.cpp:56-63
    const Factor<S> dmVInv{GEN_FRACS, FIELD_PSI, true, 0.e-6};                                          // MxEMOps.cpp:125-127
    const Factor<S> eps{kEps, FIELD_E, false, 0.0, invEps}, vol{kEpsVolAve, FIELD_PSI, false, 0.0, invEpsVolAve};
    if (name == "curlE") chain = {curlE};
    else if (name == "curlB") chain = {curlB};
    else if (name == "divB") chain = {divB};
    else if (name == "gradPsi") chain = {gradPsi};
    else if (name == "dmA" || name == "mRhs") chain = {dmA};                      // MxMagWaveOp.cpp:227-241
    else if (name == "dmL") chain = {dmL};
    else if (name == "dmVInv") chain = {dmVInv};
    else if (name == "invEps") chain = {Factor<S>{kEps, FIELD_E}};                 // MxEMOps.cpp:72-81: the simulation's own
    else if (name == "invEpsVolAve") chain = {Factor<S>{kEpsVolAve, FIELD_PSI}};
    else if (name == "curlCurl") {                                                 // MxMagWaveOp.cpp:144-153
      chain.push_back(curlE);
      if (pec) chain.push_back(dmL);
      if (withEps) chain.push_back(eps);
      chain.push_back(curlB);
    } else if (name == "gradDiv") {                                                // MxMagWaveOp.cpp:156-179
      if (pec) chain.push_back(dmA);
      chain.push_back(gradPsi);
      if (withVol) chain.push_back(vol);
      if (pec) chain.push_back(dmVInv);
      chain.push_back(divB);
      if (pec) chain.push_back(dmA);
    } else {                                                                       // scaLapl, MxMagWaveOp.cpp:208-223
      chain.push_back(divB);
      if (pec) chain.push_back(dmA);
      chain.push_back(gradPsi);
    }
    // pass 1: every factor on the rows the factor to its left references
    std::vector<Csr<S>> f(chain.size());
    struct OwnedList {
      Assembler* a; std::vector<Csr<S>>* v;
      ~OwnedList() { for (Csr<S>& m : *v) a->destroy(m); }
    } owned{this, &f};
    RowRuns rows = oneRun(r0, r1 - r0);
    for (size_t j = 0; j < chain.size(); ++j) {
      const Factor<S>& c = chain[j];
      if (c.given) {
        const int field = c.op == kEps ? FIELD_E : FIELD_PSI;
        if (c.given->mapRows != h_.f[field].nLoc || c.given->ncols != h_.f[field].nLoc)
          throw std::runtime_error("a dielectric factor handed in does not live on the simulation's maps");
        f[j] = selectRows(*c.given, rows);
        f[j].rowField = f[j].colField = field;
      } else if (c.op == kEps) {
        f[j] = buildRows<S>(rows.size(), h_.f[FIELD_E].nLoc, AtRows<InvEpsRow<S>>{InvEpsRow<S>{dSim_, hasPEC_ ? 1 : 0}, rows});
        f[j].setRuns(rows, h_.f[FIELD_E].nLoc);
        f[j].rowField = f[j].colField = FIELD_E;
        checkErr("inverse permittivity");
      } else if (c.op == kEpsVolAve) {
        f[j] = buildRows<S>(rows.size(), h_.f[FIELD_PSI].nLoc, AtRows<InvEpsVolAveRow<S>>{InvEpsVolAveRow<S>{dSim_}, rows});
        f[j].setRuns(rows, h_.f[FIELD_PSI].nLoc);
        f[j].rowField = f[j].colField = FIELD_PSI;
        checkErr("inverse permittivity");
      } else {
        f[j] = generateRows<S>(c.op, c.fracField, c.inverse, c.minFrac, rows);
      }
      if (j + 1 < chain.size()) rows = reach(f[j], f[j].runs(), f[j].colField);
    }
    // pass 2: the products, right to left
    Csr<S> m = f.back();
    f.back() = Csr<S>();
    for (size_t j = chain.size() - 1; j-- > 0;) {
      Csr<S> next;
      try {
        next = multiply(f[j], m);
      } catch (...) {
        destroy(m);
        throw;
      }
      replaceWith(m, next);
      destroy(f[j]);
    }
    if (name == "scaLapl") scale(m, scalarFrom<S>(-1.0, 0.0));
    return m;
  }

  bool complexByDefault() const { return complex_; }
  mxy::Sim* simOnExec() { return dSim_; }
  void checkErr(const char* what) {
    int e = 0;
    x_.toHost(&e, h_.err, sizeof(int));
    if (e) {
      const int zero = 0;
      x_.toExec(h_.err, &zero, sizeof(int));
      throw std::runtime_error(std::string(what) + (e == mxy::kErrStencil  ? ": a stencil left the guarded block"
                                                    : e == mxy::kErrDomain ? ": a column is not in the domain map"
                                                                           : ": a column of A has no stored row in B"));
    }
  }

 private:
  static int translateBC(int kind, int bc, int comp, int dir) {
    using namespace mxy;
    if (bc != PEC && bc != PMC) return bc;
    const bool normal = (comp == dir);
    if (kind == FIELD_PSI) return bc == PEC ? CONSTANT : ZERO;                                    // MxYeePsiField.cpp:84-93
    if (kind == FIELD_B) return bc == PEC ? (normal ? ZERO : CONSTANT) : (normal ? CONSTANT : ZERO);   // MxYeeMagFieldBase.cpp:134-163
    return bc == PEC ? (normal ? CONSTANT : ZERO) : (normal ? ZERO : CONSTANT);                   // MxYeeElecFieldBase.cpp:104-133
  }
  void pushSim() { x_.toExec(dSim_, &h_, sizeof(mxy::Sim)); }
  static void checkShape(const Shape& shape) {
    if (shape.nodes.empty()) throw std::runtime_error("empty shape");
    if (shape.depth() > kShapeMaxDepth) throw std::runtime_error("shape tree deeper than 8 levels");
  }
  ShapeNode* uploadShape(const Shape& shape) {
    ShapeNode* d = x_.template alloc<ShapeNode>(int64_t(shape.nodes.size()));
    x_.toExec(d, shape.nodes.data(), shape.nodes.size() * sizeof(ShapeNode));
    return d;
  }
  // A Bloch-consistent transfer needs complex entries unless every phase is 0 (then it equals the plain transfer bit for
  // bit), and both grids must carry the same phases.
  void checkBlochTransfer(const Assembler& from, bool realScalar) const {
    for (int i = 0; i < 3; ++i)
      if (from.phase_[i] != phase_[i]) throw std::runtime_error("Bloch transfer: the two simulations have different phase shifts");
    if (realScalar && from.complex_) throw std::runtime_error("Bloch transfer: non-zero phase shifts need a complex interpolator");
  }
  void requireSetUp() const {
    if (!setUp_) throw std::runtime_error("the simulation has not been set up (mxg_sim_setup)");
  }
  template <class S>
  void replaceWith(Csr<S>& m, Csr<S> next) {
    destroy(m);
    m = next;
  }

  X& x_;
  mxy::Sim h_;            // host copy; its pointers are executor pointers
  mxy::Sim* dSim_ = nullptr;
  Shape pec_;             // kept for the D-field fractions a later dielectric needs
  std::vector<int64_t> planeStart_[mxy::NUM_FIELDS];   // first map position of x-planes 0 .. N0 + 1, per field
  bool hasPEC_ = false, setUp_ = false, complex_ = false;
  double phase_[3] = {0.0, 0.0, 0.0};   // Bloch phase shifts per direction
};

}  // namespace mxa
