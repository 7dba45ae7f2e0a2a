// TEST INFRASTRUCTURE ONLY: the CPU oracle (oracle/mxoracle.cpp, included unchanged) plus the Bloch-consistent grid
// transfer it does not have (DESIGN.md GMG-bloch, include/mxasm.h: MXG_INTERP_BLOCH). Built by tests/bloch_oracle.py with the
// oracle's own flags (-ffp-contract=off); its matrices are the oracle's, so oracle/oracle.py's Matrix reads, transposes and
// applies them.
//
// The restatement follows the oracle's interpolator (mxo_ops.hpp, MxGridFieldInterpolator.cpp:28-122) and adds one step:
// an entry of non-zero weight whose coarse cell wraps across a PERIODIC face is multiplied by that direction's Bloch factor,
// phase from the top (cell >= N), 1 / phase from below (cell < 0), accumulated direction by direction with std::complex as
// getCompFactor accumulates its factors (MxGridField.cpp:145-190). Entries of weight 0 stay +0.
#include "../../oracle/mxoracle.cpp"

namespace {

template <class S>
Csr<S> blochInterpolator(const Field& from, const Field& to) {
  if (from.ncomp != to.ncomp) throw std::runtime_error("mxo: interpolator needs fields with equal component counts");
  Csr<S> m;
  startMatrix(m, to, from);
  const Grid& fg = *from.g;
  RowBuf<S> row;
  for (int64_t gid : to.gids) {
    I3 tcell; int comp;
    cellCompOf(to, gid, tcell, comp);
    const D3 point = to.g->nodeCoord(tcell) + to.xi[comp];
    I3 c0;
    for (int i = 0; i < 3; ++i)
      c0[i] = int(std::floor((point[i] - from.xi[comp][i] - fg.origin[i]) / fg.d[i]));
    double sum = 0.0;
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b)
        for (int c = 0; c < 2; ++c) {
          const I3 cell{c0[0] + a, c0[1] + b, c0[2] + c};
          const D3 p0 = fg.nodeCoord(cell) + from.xi[comp];
          double w = 1.0;
          for (int i = 0; i < 3; ++i) w *= 1.0 - std::fabs(point[i] - p0[i]) / fg.d[i];
          bool inRange = true;
          for (int i = 0; i < 3; ++i)
            if (cell[i] < -1 || cell[i] > fg.N[i] + 1) inRange = false;
          if (!inRange) continue;
          const int32_t l = from.lid(from.gid(comp, cell));
          if (l < 0) continue;
          if (w != 0.0) {
            cplx f(1.0, 0.0);
            for (int i = 0; i < 3; ++i) {
              if (cell[i] < 0) { if (from.lbc[comp][i] == PERIODIC) f /= from.phase[i]; }
              else if (cell[i] >= fg.N[i]) { if (from.ubc[comp][i] == PERIODIC) f *= from.phase[i]; }
            }
            row.add(l, fromFactor<S>(f) * S(w));
          } else {
            row.add(l, S(w));
          }
          sum += std::fabs(w);
        }
    if (sum > 0)
      for (auto& e : row.e) e.second = e.second / S(sum);
    row.flushInto(m);
  }
  return m;
}

}  // namespace

extern "C" {

// the Bloch-consistent transfer of field `field` from simFrom to simTo (simulations made by the oracle)
void* mxb_build_bloch_interp(void* simFrom, void* simTo, const char* field, int is_complex) {
  Mat* m = new Mat;
  m->cplx_ = is_complex != 0;
  const int rc = guard([&] {
    const Field* f = fieldOf(static_cast<Sim*>(simFrom), field);
    const Field* t = fieldOf(static_cast<Sim*>(simTo), field);
    if (m->cplx_) m->c = blochInterpolator<cplx>(*f, *t); else m->r = blochInterpolator<double>(*f, *t);
  });
  if (rc != 0) { delete m; return nullptr; }
  return m;
}

}  // extern "C"
