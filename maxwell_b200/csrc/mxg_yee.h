// Yee-grid index rules, boundary / Bloch factors, operator row generators and CRS row algebra of the operator
// assembly (SURVEY 8 f2). Everything here is a plain function of POD arguments, compiled for the device by
// mxg_asm.cu (one thread per operator row) and, unchanged, for the host by the CPU replay harness of the tests
// (tests/cpp/asm_replay.cpp) -- the replay pins the logic without a GPU; only rounding could differ, and the
// translation unit is built with -fmad=false so a*b+c stays two roundings as on the reference's host.
//
// Reference files (paths relative to bauerca/maxwell src/): MxGrid.h:96-128 (cell <-> global), MxGridField.cpp:41-77
// (useCompInMap), :80-142 (getInteriorComp), :145-190 (getCompFactor), :256-297 (setMap), MxGridField.hpp:142-145
// (component GID), MxYeeFitBField.cpp:63-90, MxYeeFitEField.cpp:53-98, MxYeePsiField.cpp:100-124 (Dey-Mittra
// overrides), MxYeeDeyMittraCurlE.cpp:117-178, CurlB.cpp:113-169, DivB.cpp:157-200, GradPsi.cpp:23-84,
// Fracs.cpp:30-131 (generators), MxCrsMatrix.cpp:84-117,358-430 (purge, multiply, add).
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define MXY_HD __host__ __device__ __forceinline__
#else
#define MXY_HD inline
#endif

namespace mxy {

enum BCType { PERIODIC = 0, ZERO = 1, CONSTANT = 2, PEC = 3, PMC = 4 };
// B, E and psi carry DOF maps; D (the dual-face field of the dielectric update, MxYeeFitDField) shares E's map and exists
// only to hold face fractions and boundary factors at the E positions
enum FieldKind { FIELD_B = 0, FIELD_E = 1, FIELD_PSI = 2, NUM_FIELDS = 3, FIELD_D = 3, NUM_ALL_FIELDS = 4 };
constexpr int kMaxDielectrics = 4;
enum FactorAction { ACT_NONE = 0, ACT_DIV = 1, ACT_MUL = 2, ACT_NEG = 3, ACT_ZERO = 4 };

// complex scalar: (re, im), bit-compatible with std::complex<double>
struct Cx {
  double re, im;
};
MXY_HD double mulS(double a, double b) { return a * b; }
MXY_HD Cx mulS(Cx a, Cx b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
MXY_HD double addS(double a, double b) { return a + b; }
MXY_HD Cx addS(Cx a, Cx b) { return {a.re + b.re, a.im + b.im}; }
template <class S> MXY_HD S fromParts(double re, double im);
template <> MXY_HD double fromParts<double>(double re, double) { return re; }   // MxUtil.hpp:58-62: real builds keep Re
template <> MXY_HD Cx fromParts<Cx>(double re, double im) { return {re, im}; }
MXY_HD double absD(double v) { return v < 0.0 ? -v : v; }
MXY_HD bool survivesPurge(double v) { return absD(v) > 1.e-12; }                  // MxCrsMatrix.cpp:84-117
MXY_HD bool survivesPurge(Cx v) { return absD(v.re) > 1.e-12 || absD(v.im) > 1.e-12; }

struct Grid {
  int N[3];
  double origin[3], d[3];
};

struct Field {
  int kind, ncomp;
  double xi[3][3];          // cell-relative component positions
  int lbc[3][3], ubc[3][3]; // per component and direction, already translated from PEC / PMC walls
  double dmFrac;
  int regionSet;            // a PEC shape restricts the map
  int literalUpperPeriodicE;
  const double* region;     // PEC fractions on the guarded block (cells -1 .. N+1), [cell][comp]
  const int32_t* lidOf;     // dense GID -> position in the map (-1: not a DOF)
  const int64_t* gids;      // the map, ascending
  int64_t nLoc;
  // Boundary / Bloch factor of every per-direction action triple, evaluated once on the host in the reference's
  // order of operations (complex division included), so device rows pick the very same doubles.
  double facRe[125], facIm[125];
};

// MxDielectric: a shape with a (possibly anisotropic, possibly complex) permittivity tensor; fractions of the shape on the
// E edges, the dual D faces and the psi cells of the guarded block (MxEMSim.cpp:134-148)
struct DielectricRep {
  const double* fracE;
  const double* fracD;
  const double* fracPsi;
  const void* shape;        // flattened shape nodes on the executor (mxg_shape.h), for the interface normal
  double epsRe[9], epsIm[9];
  int isDiag;
};

struct Sim {
  Grid g;
  Field f[NUM_ALL_FIELDS];
  int* err;                 // set to non-zero by row functions that meet an impossible index
  int numDiel;
  DielectricRep diel[kMaxDielectrics];
};

// ---- indexing -------------------------------------------------------------------------------------------------
MXY_HD int64_t cellToGlobal(const Grid& g, const int c[3]) {     // MxGrid.h:96-114
  int64_t res = 0, factor = 1;
  for (int i = 2; i >= 0; --i) {
    const int ni = g.N[i] + 1;
    int v = c[i];
    if (v >= ni) v -= ni; else if (v < 0) v += ni;
    res += int64_t(v) * factor;
    factor *= ni;
  }
  return res;
}
MXY_HD void globalToCell(const Grid& g, int64_t idx, int c[3]) {
  int64_t factor = 1;
  for (int i = 2; i >= 0; --i) {
    const int ni = g.N[i] + 1;
    c[i] = int((idx / factor) % ni);
    factor *= ni;
  }
}
MXY_HD int64_t numNodes(const Grid& g) { return int64_t(g.N[0] + 1) * (g.N[1] + 1) * (g.N[2] + 1); }
MXY_HD int64_t numFullCells(const Grid& g) { return int64_t(g.N[0] + 3) * (g.N[1] + 3) * (g.N[2] + 3); }
// guarded block index; -1 when the cell lies outside cells -1 .. N+1
MXY_HD int64_t fullIndex(const Grid& g, const int c[3]) {
  int64_t res = 0, factor = 1;
  for (int i = 2; i >= 0; --i) {
    if (c[i] < -1 || c[i] >= g.N[i] + 2) return -1;
    res += int64_t(c[i] + 1) * factor;
    factor *= (g.N[i] + 3);
  }
  return res;
}
MXY_HD void fullToCell(const Grid& g, int64_t i, int c[3]) {
  const int n1 = g.N[1] + 3, n2 = g.N[2] + 3;
  c[2] = int(i % n2) - 1;
  c[1] = int((i / n2) % n1) - 1;
  c[0] = int(i / (int64_t(n2) * n1)) - 1;
}

MXY_HD double regionFrac(const Sim& s, const Field& f, int comp, const int cell[3]) {
  if (!f.region) return 1.0;
  const int64_t fi = fullIndex(s.g, cell);
  if (fi < 0) { if (s.err) *s.err = 1; return 1.0; }
  return f.region[comp + f.ncomp * fi];
}

// MxGridField.cpp:80-142 (its "case 1" is always overwritten by "case 2")
MXY_HD void interior(const Grid& g, const Field& f, int comp, const int cell[3], int nc[3]) {
  for (int i = 0; i < 3; ++i) {
    const int n = g.N[i];
    const bool onLower = (f.xi[comp][i] == 0.0);
    nc[i] = cell[i];
    if (cell[i] < 0) {
      nc[i] = (f.lbc[comp][i] == PERIODIC) ? n + cell[i] : -cell[i] - 1;
    } else if (cell[i] == n && onLower) {
      if (f.ubc[comp][i] == PERIODIC) nc[i] = 0;
    } else if (cell[i] >= n && onLower) {
      nc[i] = (f.ubc[comp][i] == PERIODIC) ? cell[i] - n : n - (cell[i] - n);
    } else if (cell[i] >= n) {
      nc[i] = (f.ubc[comp][i] == PERIODIC) ? cell[i] - n : n - (cell[i] - n + 1);
    }
  }
}
MXY_HD int64_t gidOf(const Grid& g, const Field& f, int comp, const int cell[3]) {   // MxGridField.hpp:142-145
  int nc[3];
  interior(g, f, comp, cell, nc);
  return comp + f.ncomp * cellToGlobal(g, nc);
}

// MxGridField.cpp:41-77
MXY_HD bool baseUse(const Sim& s, const Field& f, int comp, const int cell[3]) {
  if (f.regionSet && regionFrac(s, f, comp, cell) == 0.0) return false;
  for (int i = 0; i < 3; ++i) {
    const int n = s.g.N[i];
    const double x = f.xi[comp][i];
    if (cell[i] == 0 && x == 0.0) {
      if (f.lbc[comp][i] == ZERO) return false;
    } else if (cell[i] == n && x > 0.0) {
      return false;
    } else if (cell[i] == n && x == 0.0) {
      if (f.ubc[comp][i] == ZERO || f.ubc[comp][i] == PERIODIC) return false;
    }
  }
  return true;
}
MXY_HD bool useB(const Sim& s, int comp, const int cell[3]) {       // MxYeeFitBField.cpp:63-80
  const Field& B = s.f[FIELD_B];
  for (int c = 0; c < 3; ++c)
    if (baseUse(s, B, c, cell)) return true;
  bool res = baseUse(s, B, comp, cell);
  if (B.regionSet && regionFrac(s, B, comp, cell) < B.dmFrac) res = false;
  return res;
}
MXY_HD bool useComp(const Sim& s, int kind, int comp, const int cellIn[3]) {
  int cell[3] = {cellIn[0], cellIn[1], cellIn[2]};
  if (kind == FIELD_B) return useB(s, comp, cell);
  const Field& f = s.f[kind];
  if (!baseUse(s, f, comp, cell)) return false;
  if (kind == FIELD_E) {                                           // MxYeeFitEField.cpp:53-88
    const int c2 = (comp + 1) % 3, c3 = (comp + 2) % 3;
    if (!useB(s, c2, cell)) return false;
    cell[c3]--;
    if (!useB(s, c2, cell)) return false;
    cell[c3]++;
    if (!useB(s, c3, cell)) return false;
    cell[c2]--;
    if (!useB(s, c3, cell)) return false;
    return true;
  }
  for (int i = 0; i < 3; ++i) {                                     // MxYeePsiField.cpp:100-114
    if (useB(s, i, cell)) return true;
    cell[i]++;
    if (useB(s, i, cell)) return true;
    cell[i]--;
  }
  return false;
}

// MxGridField.cpp:145-190: which of {nothing, / phase, * phase, * -1, * 0} each direction applies
MXY_HD int factorCode(const Grid& g, const Field& f, int comp, const int cell[3]) {
  int code = 0;
  for (int i = 0; i < 3; ++i) {
    const int n = g.N[i];
    const double x = f.xi[comp][i];
    const int lo = f.lbc[comp][i], up = f.ubc[comp][i];
    int act = ACT_NONE;
    if (cell[i] < 0) {
      if (lo == PERIODIC) act = ACT_DIV;
      else if (lo == ZERO) act = ACT_NEG;
    } else if (cell[i] == 0 && x == 0.0) {
      if (lo == ZERO) act = ACT_ZERO;
    } else if (cell[i] == n && x == 0.0) {
      if (up == PERIODIC) act = ACT_MUL;
      else if (up == ZERO) act = ACT_ZERO;
    } else if (cell[i] >= n) {
      if (up == PERIODIC) act = ACT_MUL;
      else if (up == ZERO) act = ACT_NEG;
    }
    code = code * 5 + act;
  }
  return code;
}
// MxYeeFitBField.cpp:82-90, MxYeeFitEField.cpp:90-98, MxYeePsiField.cpp:116-124. Returns false for a zero factor.
MXY_HD bool factorOf(const Sim& s, int kind, int comp, const int cell[3], double& re, double& im) {
  const Field& f = s.f[kind];
  re = 0.0; im = 0.0;
  if (kind == FIELD_B && f.regionSet && regionFrac(s, f, comp, cell) < f.dmFrac) return false;
  if (f.regionSet && regionFrac(s, f, comp, cell) == 0.0) return false;
  const int code = factorCode(s.g, f, comp, cell);
  if (kind == FIELD_E || kind == FIELD_PSI) {
    // The reference tests useCompInMap on the un-wrapped cell; by default the wrapped one is tested so the
    // wrap-around entry of a PERIODIC upper boundary survives (DESIGN.md R13).
    int c[3] = {cell[0], cell[1], cell[2]};
    if (!f.literalUpperPeriodicE)
      for (int i = 0; i < 3; ++i)
        if (c[i] >= s.g.N[i] && f.ubc[comp][i] == PERIODIC && f.lbc[comp][i] == PERIODIC) c[i] -= s.g.N[i];
    if (!useComp(s, kind, comp, c)) return false;
  }
  re = f.facRe[code];
  im = f.facIm[code];
  return !(re == 0.0 && im == 0.0);
}

// ---- row buffers ------------------------------------------------------------------------------------------------
// Epetra semantics of InsertGlobalValues + FillComplete (MxCrsMatrix.cpp:122-143,325-342): ascending local column,
// duplicate insertions summed in insertion order, explicit zeros kept.
template <class S>
MXY_HD int flushRow(int n, int32_t* cols, S* vals) {
  for (int i = 1; i < n; ++i) {            // stable insertion sort by column
    const int32_t c = cols[i];
    const S v = vals[i];
    int j = i - 1;
    while (j >= 0 && cols[j] > c) { cols[j + 1] = cols[j]; vals[j + 1] = vals[j]; --j; }
    cols[j + 1] = c;
    vals[j + 1] = v;
  }
  int o = 0;
  for (int i = 0; i < n;) {
    S sum = vals[i];
    int j = i + 1;
    while (j < n && cols[j] == cols[i]) sum = addS(sum, vals[j++]);
    cols[o] = cols[i];
    vals[o] = sum;
    ++o;
    i = j;
  }
  return o;
}

MXY_HD void cellCompOf(const Sim& s, const Field& f, int64_t gid, int cell[3], int& comp) {
  comp = int(gid % f.ncomp);                           // MxGridFieldIter.hpp:34,66-70
  globalToCell(s.g, gid / f.ncomp, cell);
}

// one candidate entry: column field `kind`, component, cell, coefficient
template <class S>
MXY_HD void addEntry(const Sim& s, int kind, int comp, const int cell[3], double coef, int& n, int32_t* cols, S* vals) {
  double re, im;
  if (!factorOf(s, kind, comp, cell, re, im)) return;
  const Field& f = s.f[kind];
  const int32_t l = f.lidOf[gidOf(s.g, f, comp, cell)];
  if (l < 0) { if (s.err) *s.err = 2; return; }        // an operator may not reference a column outside the domain map
  cols[n] = l;
  vals[n] = mulS(fromParts<S>(re, im), fromParts<S>(coef, 0.0));
  ++n;
}

enum GenOp { GEN_CURL_E = 0, GEN_CURL_B = 1, GEN_DIV_B = 2, GEN_GRAD_PSI = 3, GEN_FRACS = 4 };
constexpr int kGenMaxRow = 8;

// Row `row` of a generated operator; returns the entry count (<= kGenMaxRow), entries sorted and merged.
template <class S>
struct GenRow {
  static constexpr int kMax = kGenMaxRow;
  const Sim* sim;
  int op;
  int fracField;      // GEN_FRACS: which field
  int fracInverse;
  double fracMin;
  MXY_HD int operator()(int64_t row, int32_t* cols, S* vals) const {
    const Sim& s = *sim;
    const Grid& g = s.g;
    int n = 0, cell[3], c0;
    if (op == GEN_CURL_E) {                            // MxYeeDeyMittraCurlE.cpp:117-178
      const Field& B = s.f[FIELD_B];
      cellCompOf(s, B, B.gids[row], cell, c0);
      const int c1 = (c0 + 1) % 3, c2 = (c0 + 2) % 3;
      double re, im;
      if (factorOf(s, FIELD_B, c0, cell, re, im)) {
        const double i1 = 1 / g.d[c1], i2 = 1 / g.d[c2];
        cell[c1]++; addEntry<S>(s, FIELD_E, c2, cell, i1, n, cols, vals);
        cell[c1]--; addEntry<S>(s, FIELD_E, c2, cell, -i1, n, cols, vals);
        cell[c2]++; addEntry<S>(s, FIELD_E, c1, cell, -i2, n, cols, vals);
        cell[c2]--; addEntry<S>(s, FIELD_E, c1, cell, i2, n, cols, vals);
      }
    } else if (op == GEN_CURL_B) {                     // MxYeeDeyMittraCurlB.cpp:113-169
      const Field& E = s.f[FIELD_E];
      cellCompOf(s, E, E.gids[row], cell, c0);
      const int c1 = (c0 + 1) % 3, c2 = (c0 + 2) % 3;
      const double i1 = 1 / g.d[c1], i2 = 1 / g.d[c2];
      addEntry<S>(s, FIELD_B, c2, cell, i1, n, cols, vals);
      cell[c1]--; addEntry<S>(s, FIELD_B, c2, cell, -i1, n, cols, vals);
      cell[c1]++; addEntry<S>(s, FIELD_B, c1, cell, -i2, n, cols, vals);
      cell[c2]--; addEntry<S>(s, FIELD_B, c1, cell, i2, n, cols, vals);
    } else if (op == GEN_DIV_B) {                      // MxYeeDeyMittraDivB.cpp:157-200
      const Field& P = s.f[FIELD_PSI];
      cellCompOf(s, P, P.gids[row], cell, c0);
      for (int c = 0; c < 3; ++c) {
        cell[c]++; addEntry<S>(s, FIELD_B, c, cell, 1.0 / g.d[c], n, cols, vals);
        cell[c]--; addEntry<S>(s, FIELD_B, c, cell, -1.0 / g.d[c], n, cols, vals);
      }
    } else if (op == GEN_GRAD_PSI) {                   // MxYeeDeyMittraGradPsi.cpp:23-84
      const Field& B = s.f[FIELD_B];
      cellCompOf(s, B, B.gids[row], cell, c0);
      double re, im;
      if (factorOf(s, FIELD_B, c0, cell, re, im)) {
        const double inv = 1.0 / g.d[c0];
        addEntry<S>(s, FIELD_PSI, 0, cell, inv, n, cols, vals);
        cell[c0]--; addEntry<S>(s, FIELD_PSI, 0, cell, -inv, n, cols, vals);
      }
    } else {                                           // MxYeeDeyMittraFracs.cpp:30-131: zeros are stored
      const Field& F = s.f[fracField];
      cellCompOf(s, F, F.gids[row], cell, c0);
      double v = regionFrac(s, F, c0, cell);
      if (!fracInverse) {
        if (v != 0 && v < fracMin) v = fracMin;
      } else {
        if (v == 0) {}
        else if (v < fracMin) v = 1.0 / fracMin;
        else v = 1.0 / v;
      }
      cols[0] = int32_t(row);
      vals[0] = fromParts<S>(v, 0.0);
      return 1;
    }
    return flushRow<S>(n, cols, vals);
  }
};

// ---- CRS row algebra --------------------------------------------------------------------------------------------
// The rows a CRS matrix stores: at most two runs of positions in its row field's map, stored one after the other
// (a whole-map matrix: one run from 0). Two runs arise on periodic-x grids, where a slab's stencils reach the planes on
// the far side of the wrap.
struct RowRuns {
  int64_t begin[2], count[2];
  MXY_HD int64_t size() const { return count[0] + count[1]; }
  MXY_HD int64_t pos(int64_t i) const { return i < count[0] ? begin[0] + i : begin[1] + (i - count[0]); }   // stored -> map
  MXY_HD int64_t find(int64_t k) const {                                                                   // map -> stored, -1
    if (k >= begin[0] && k - begin[0] < count[0]) return k - begin[0];
    if (k >= begin[1] && k - begin[1] < count[1]) return count[0] + (k - begin[1]);
    return -1;
  }
};
MXY_HD RowRuns oneRun(int64_t begin, int64_t count) { return {{begin, 0}, {count, 0}}; }

template <class S>
struct CsrView {
  int64_t nrows, ncols;
  const int64_t* rowptr;
  const int32_t* col;
  const S* val;
  RowRuns runs;             // which map positions the stored rows are
};

constexpr int kErrStencil = 1, kErrDomain = 2, kErrNotStored = 3;   // codes of Sim::err

// Upper bound of the row length of A * B (before merging): the table size the product kernel is instantiated with.
// B is read through its stored runs; a column of A that B does not store sets kErrNotStored.
template <class S>
struct ProductBound {
  CsrView<S> A, B;
  int* err;
  MXY_HD int operator()(int64_t i) const {
    int64_t n = 0;
    for (int64_t p = A.rowptr[i]; p < A.rowptr[i + 1]; ++p) {
      const int64_t k = B.runs.find(A.col[p]);
      if (k < 0) { *err = kErrNotStored; continue; }
      n += B.rowptr[k + 1] - B.rowptr[k];
    }
    return n > 0x7fffffff ? 0x7fffffff : int(n);
  }
};

// Row i of A * B with the accumulation order of EpetraExt::MatrixMatrix::Multiply as the reference drives it
// (MxCrsMatrix.cpp:358-382): C(i,j) sums over A's stored row order, cancellation zeros are kept.
template <class S, int MAXC>
struct ProductRow {
  static constexpr int kMax = MAXC;
  CsrView<S> A, B;
  int* err;
  MXY_HD int operator()(int64_t i, int32_t* cols, S* vals) const {
    int n = 0;
    for (int64_t p = A.rowptr[i]; p < A.rowptr[i + 1]; ++p) {
      const int64_t k = B.runs.find(A.col[p]);
      if (k < 0) { *err = kErrNotStored; continue; }
      const S a = A.val[p];
      for (int64_t q = B.rowptr[k]; q < B.rowptr[k + 1]; ++q) {
        const int32_t j = B.col[q];
        const S prod = mulS(a, B.val[q]);
        int t = 0;
        while (t < n && cols[t] != j) ++t;
        if (t < n) vals[t] = addS(vals[t], prod);
        else if (n < MAXC) { cols[n] = j; vals[n] = prod; ++n; }
      }
    }
    for (int i2 = 1; i2 < n; ++i2) {       // columns are unique now: any sort gives the same row
      const int32_t c = cols[i2];
      const S v = vals[i2];
      int j = i2 - 1;
      while (j >= 0 && cols[j] > c) { cols[j + 1] = cols[j]; vals[j + 1] = vals[j]; --j; }
      cols[j + 1] = c;
      vals[j + 1] = v;
    }
    return n;
  }
};

// Row i of sa*A + sb*B on the union pattern (EpetraExt::MatrixMatrix::Add; MxCrsMatrix.cpp:401-430); optionally
// drops entries with magnitude <= 1e-12 (MxCrsMatrix.cpp:84-117) in the same pass.
template <class S, int MAXC>
struct SumRow {
  static constexpr int kMax = MAXC;
  CsrView<S> A, B;
  S sa, sb;
  int purge;
  MXY_HD int operator()(int64_t i, int32_t* cols, S* vals) const {
    int64_t p = A.rowptr[i], pe = A.rowptr[i + 1], q = B.rowptr[i], qe = B.rowptr[i + 1];
    int n = 0;
    while (p < pe || q < qe) {
      int32_t c;
      S v;
      if (q >= qe || (p < pe && A.col[p] < B.col[q])) { c = A.col[p]; v = mulS(sa, A.val[p]); ++p; }
      else if (p >= pe || B.col[q] < A.col[p]) { c = B.col[q]; v = mulS(sb, B.val[q]); ++q; }
      else { c = A.col[p]; v = addS(mulS(sa, A.val[p]), mulS(sb, B.val[q])); ++p; ++q; }
      if (purge && !survivesPurge(v)) continue;
      if (n < MAXC) { cols[n] = c; vals[n] = v; ++n; }
    }
    return n;
  }
};

// Row i of A with small entries dropped.
template <class S, int MAXC>
struct PurgeRow {
  static constexpr int kMax = MAXC;
  CsrView<S> A;
  MXY_HD int operator()(int64_t i, int32_t* cols, S* vals) const {
    int n = 0;
    for (int64_t p = A.rowptr[i]; p < A.rowptr[i + 1]; ++p)
      if (survivesPurge(A.val[p]) && n < MAXC) { cols[n] = A.col[p]; vals[n] = A.val[p]; ++n; }
    return n;
  }
};

// A row generator evaluated on the stored rows `runs` of its map: stored row i is map row runs.pos(i).
template <class Fn>
struct AtRows {
  static constexpr int kMax = Fn::kMax;
  Fn fn;
  RowRuns runs;
  template <class S>
  MXY_HD int operator()(int64_t i, int32_t* cols, S* vals) const { return fn(runs.pos(i), cols, vals); }
};

// Which x-planes of the column field the map rows `over` of A reference: flag[plane] = 1 (GIDs are x-major, so a plane
// is one run of the column field's map). `over` must be stored in A.
template <class S>
struct PlaneFlags {
  CsrView<S> A;
  RowRuns over;
  const int64_t* colGids;   // column field map
  int64_t planeGids;        // GIDs per x-plane: ncomp (N1 + 1) (N2 + 1)
  int32_t* flag;
  MXY_HD void operator()(int64_t i) const {
    const int64_t s = A.runs.find(over.pos(i));
    for (int64_t p = A.rowptr[s]; p < A.rowptr[s + 1]; ++p) flag[colGids[A.col[p]] / planeGids] = 1;
  }
};

// How many entries of stored row i of A have a column that B does not store (checked before a product reads B).
template <class S>
struct MissingCols {
  CsrView<S> A;
  RowRuns bRuns;
  MXY_HD int operator()(int64_t i) const {
    int n = 0;
    for (int64_t p = A.rowptr[i]; p < A.rowptr[i + 1]; ++p) n += bRuns.find(A.col[p]) < 0 ? 1 : 0;
    return n;
  }
};

// Copy of the map rows `over` of A (which stores them): row lengths, then entries.
template <class S>
struct SelectCount {
  CsrView<S> A;
  RowRuns over;
  int32_t* count;
  MXY_HD void operator()(int64_t i) const {
    const int64_t s = A.runs.find(over.pos(i));
    count[i] = int32_t(A.rowptr[s + 1] - A.rowptr[s]);
  }
};
template <class S>
struct SelectFill {
  CsrView<S> A;
  RowRuns over;
  const int64_t* rowptr;
  int32_t* col;
  S* val;
  MXY_HD void operator()(int64_t i) const {
    const int64_t s = A.runs.find(over.pos(i));
    int64_t o = rowptr[i];
    for (int64_t p = A.rowptr[s]; p < A.rowptr[s + 1]; ++p, ++o) { col[o] = A.col[p]; val[o] = A.val[p]; }
  }
};

// First map position of every x-plane: out[p] = lower bound of p * planeGids in the ascending map (p = 0 .. N0 + 1).
struct PlaneStart {
  const int64_t* gids;
  int64_t n, planeGids;
  int64_t* out;
  MXY_HD void operator()(int64_t p) const {
    const int64_t key = p * planeGids;
    int64_t lo = 0, hi = n;
    while (lo < hi) {
      const int64_t mid = lo + (hi - lo) / 2;
      if (gids[mid] < key) lo = mid + 1; else hi = mid;
    }
    out[p] = lo;
  }
};

// pass 1 / pass 2 of every row-generated CRS matrix
template <class S, class RowFn>
struct CountRows {
  RowFn fn;
  int32_t* count;
  MXY_HD void operator()(int64_t i) const {
    int32_t cols[RowFn::kMax];
    S vals[RowFn::kMax];
    count[i] = fn(i, cols, vals);
  }
};
template <class S, class RowFn>
struct FillRows {
  RowFn fn;
  const int64_t* rowptr;
  int32_t* col;
  S* val;
  MXY_HD void operator()(int64_t i) const {
    int32_t cols[RowFn::kMax];
    S vals[RowFn::kMax];
    const int n = fn(i, cols, vals);
    const int64_t o = rowptr[i];
    for (int k = 0; k < n; ++k) { col[o + k] = cols[k]; val[o + k] = vals[k]; }
  }
};

// ---- grid transfers and transposition --------------------------------------------------------------------------------
MXY_HD double divReal(double v, double s) { return v / s; }
MXY_HD Cx divReal(Cx v, double s) { return {v.re / s, v.im / s}; }   // what (v + 0i) / (s + 0i) evaluates to for s > 0
MXY_HD double conjS(double v) { return v; }
MXY_HD Cx conjS(Cx v) { return {v.re, -v.im}; }
MXY_HD double floorD(double v) {
#if defined(__CUDA_ARCH__)
  return ::floor(v);
#else
  return __builtin_floor(v);
#endif
}
MXY_HD int32_t fetchInc(int32_t* p) {
#if defined(__CUDA_ARCH__)
  return atomicAdd(p, 1);
#else
  return __atomic_fetch_add(p, 1, __ATOMIC_RELAXED);
#endif
}

// MxGridFieldInterpolator.cpp:28-65 (stencil), :68-122 (insertion, row-sum normalisation): (tri)linear interpolation of
// a field of the `from` grid at the component positions of the `to` grid. Entries whose column is not a DOF are
// dropped, then the row is divided by the sum of the magnitudes of what is left. (The reference's unset stencil point
// and never-zeroed row-sum accumulator are not reproduced, DESIGN.md R12.)
//
// bloch != 0 (DESIGN.md GMG-bloch, not in the reference): a stencil cell that wraps across a PERIODIC face of the coarse
// grid carries that direction's Bloch factor, e^{+i phi} from the top (cell >= N, ACT_MUL) and e^{-i phi} from below
// (cell < 0, ACT_DIV), looked up in the coarse field's factor table, so that P maps a coarse Bloch-periodic field onto
// the fine one. PEC / PMC images get no factor here. The row-sum normalisation still uses the weights, and entries of
// weight 0 keep the value +0 (a factor would give them the signs of its parts).
template <class S>
struct InterpRow {
  static constexpr int kMax = 8;
  const Sim* from;
  const Sim* to;
  int kind;
  int bloch;
  MXY_HD int operator()(int64_t row, int32_t* cols, S* vals) const {
    const Sim& sf = *from;
    const Sim& st = *to;
    const Field& ff = sf.f[kind];
    const Field& tf = st.f[kind];
    int tcell[3], comp;
    cellCompOf(st, tf, tf.gids[row], tcell, comp);
    double point[3];
    int c0[3];
    for (int i = 0; i < 3; ++i) {
      point[i] = (st.g.origin[i] + double(tcell[i]) * st.g.d[i]) + tf.xi[comp][i];
      c0[i] = int(floorD((point[i] - ff.xi[comp][i] - sf.g.origin[i]) / sf.g.d[i]));
    }
    double sum = 0.0;
    int n = 0;
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b)
        for (int c = 0; c < 2; ++c) {
          const int cell[3] = {c0[0] + a, c0[1] + b, c0[2] + c};
          double w = 1.0;
          bool inRange = true;
          for (int i = 0; i < 3; ++i) {
            const double p0 = (sf.g.origin[i] + double(cell[i]) * sf.g.d[i]) + ff.xi[comp][i];
            w *= 1.0 - absD(point[i] - p0) / sf.g.d[i];
            if (cell[i] < -1 || cell[i] > sf.g.N[i] + 1) inRange = false;
          }
          if (!inRange) continue;
          const int32_t l = ff.lidOf[gidOf(sf.g, ff, comp, cell)];
          if (l < 0) continue;
          cols[n] = l;
          vals[n] = fromParts<S>(w, 0.0);
          if (bloch && w != 0.0) {            // a zero weight stays (+0, +0), whatever the factor's signs
            int code = 0;
            for (int i = 0; i < 3; ++i) {
              int act = ACT_NONE;
              if (cell[i] < 0) { if (ff.lbc[comp][i] == PERIODIC) act = ACT_DIV; }
              else if (cell[i] >= sf.g.N[i]) { if (ff.ubc[comp][i] == PERIODIC) act = ACT_MUL; }
              code = code * 5 + act;
            }
            vals[n] = mulS(fromParts<S>(ff.facRe[code], ff.facIm[code]), vals[n]);
          }
          ++n;
          sum += absD(w);
        }
    if (sum > 0)
      for (int e = 0; e < n; ++e) vals[e] = divReal(vals[e], sum);
    return flushRow<S>(n, cols, vals);
  }
};

// (conjugate) transpose in three passes: column counts, scattered fill, then every row sorted by column so that the
// result does not depend on the order in which threads claimed their slots. Only the columns of the window [c0, c1)
// become rows (row j - c0); the columns of the result are A's map rows (A.runs.pos of the stored row).
struct TransposeCount {
  const int32_t* col;
  int32_t c0, c1;
  int32_t* count;
  MXY_HD void operator()(int64_t q) const {
    const int32_t j = col[q];
    if (j >= c0 && j < c1) fetchInc(count + (j - c0));
  }
};
template <class S>
struct TransposeFill {
  CsrView<S> A;
  int32_t c0, c1;
  const int64_t* tptr;
  int32_t* fill;
  int32_t* tcol;
  S* tval;
  MXY_HD void operator()(int64_t i) const {
    for (int64_t p = A.rowptr[i]; p < A.rowptr[i + 1]; ++p) {
      const int32_t j = A.col[p];
      if (j < c0 || j >= c1) continue;
      const int64_t pos = tptr[j - c0] + fetchInc(fill + (j - c0));
      tcol[pos] = int32_t(A.runs.pos(i));
      tval[pos] = conjS(A.val[p]);
    }
  }
};
// entries of stored row first + i of A whose column lies in [c0, c1)
template <class S>
struct WindowHits {
  CsrView<S> A;
  int64_t first;
  int32_t c0, c1;
  MXY_HD int operator()(int64_t i) const {
    int n = 0;
    for (int64_t p = A.rowptr[first + i]; p < A.rowptr[first + i + 1]; ++p) n += (A.col[p] >= c0 && A.col[p] < c1) ? 1 : 0;
    return n;
  }
};
template <class S>
struct SortRowInPlace {
  const int64_t* rowptr;
  int32_t* col;
  S* val;
  MXY_HD void operator()(int64_t i) const {
    const int64_t b = rowptr[i], e = rowptr[i + 1];
    for (int64_t k = b + 1; k < e; ++k) {
      const int32_t c = col[k];
      const S v = val[k];
      int64_t j = k - 1;
      while (j >= b && col[j] > c) { col[j + 1] = col[j]; val[j + 1] = val[j]; --j; }
      col[j + 1] = c;
      val[j + 1] = v;
    }
  }
};

// DOF flags of a field over the in-range cells (MxGridField.cpp:256-297: x slow .. z fast, components inner)
struct MapFlags {
  const Sim* sim;
  int kind;
  int32_t* flag;
  MXY_HD void operator()(int64_t i) const {
    const Sim& s = *sim;
    const int ncomp = s.f[kind].ncomp;
    int cell[3];
    globalToCell(s.g, i / ncomp, cell);
    flag[i] = useComp(s, kind, int(i % ncomp), cell) ? 1 : 0;
  }
};
// lidOf / gids from the scanned flags
struct MapFill {
  const int32_t* flag;
  const int64_t* offset;
  int32_t* lidOf;
  int64_t* gids;
  MXY_HD void operator()(int64_t i) const {
    if (flag[i]) { lidOf[i] = int32_t(offset[i]); gids[offset[i]] = i; }
    else lidOf[i] = -1;
  }
};

}  // namespace mxy
