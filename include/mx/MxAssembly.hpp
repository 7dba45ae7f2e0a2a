// C++ shims over the operator-assembly C ABI (include/mxasm.h) with the shape of the reference's set-up classes:
// MxShape and its subclasses (src/MxShape.hpp, MxCylinder.hpp, ...), MxEMSim (src/MxEMSim.cpp:54-199) and the CRS algebra
// of MxCrsMatrix / MxUtil (src/MxCrsMatrix.cpp:84-117,358-430, MxUtil.cpp:318-371). Header-only; link with -lmxgpu.
//
//   MxShape cyl = MxShape::cylinder(0.4, z, o), caps = MxShape::slab(0.8, z, o);
//   MxShape cav = MxShape::intersection({&cyl, &caps});
//   MxEMSim sim(comm, {256, 256, 256}, origin, size);
//   sim.setPEC(cav);
//   sim.setup();
//   auto bmap = sim.getMap("bfield");
//   auto A = sim.getOp("vecLapl").fillComplete<double>(bmap, bmap);      // an MxCrsMatrix<double>, ready to apply
#pragma once
#include <array>
#include <initializer_list>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "MxLinAlg.hpp"
#include "mxasm.h"

namespace mx {
typedef std::array<double, 3> Vec3;
}  // namespace mx

// CSG solid (f > 0 inside). Composites copy their parts.
class MxShape {
 public:
  MxShape() = default;
  ~MxShape() { if (h_) mxg_shape_destroy(h_); }
  MxShape(MxShape&& o) noexcept : h_(o.h_) { o.h_ = nullptr; }
  MxShape& operator=(MxShape&& o) noexcept {
    if (this != &o) { if (h_) mxg_shape_destroy(h_); h_ = o.h_; o.h_ = nullptr; }
    return *this;
  }
  MxShape(const MxShape&) = delete;
  MxShape& operator=(const MxShape&) = delete;

  static MxShape cylinder(double radius, const mx::Vec3& axis, const mx::Vec3& loc) {               // MxCylinder.hpp:34-40
    MxShape s; mx::check(mxg_shape_cylinder(radius, axis.data(), loc.data(), &s.h_)); return s;
  }
  static MxShape sphere(double radius, const mx::Vec3& loc) {                                    // MxSphere.hpp:31-33
    MxShape s; mx::check(mxg_shape_sphere(radius, loc.data(), &s.h_)); return s;
  }
  static MxShape halfSpace(const mx::Vec3& pointInPlane, const mx::Vec3& normal) {                   // MxHalfSpace.hpp:31-33
    MxShape s; mx::check(mxg_shape_halfspace(pointInPlane.data(), normal.data(), &s.h_)); return s;
  }
  static MxShape slab(double thickness, const mx::Vec3& normal, const mx::Vec3& loc) {               // MxSlab.hpp:33-39
    MxShape s; mx::check(mxg_shape_slab(thickness, normal.data(), loc.data(), &s.h_)); return s;
  }
  static MxShape ellipsoid(const mx::Vec3& loc, const mx::Vec3& axes) {                              // MxEllipsoid.hpp:31-33
    MxShape s; mx::check(mxg_shape_ellipsoid(loc.data(), axes.data(), &s.h_)); return s;
  }
  static MxShape torus(double majorRadius, double minorRadius, const mx::Vec3& axis, const mx::Vec3& loc) {   // MxTorus.hpp:31-37
    MxShape s; mx::check(mxg_shape_torus(majorRadius, minorRadius, axis.data(), loc.data(), &s.h_)); return s;
  }
  static MxShape cone(double angle, const mx::Vec3& axis, const mx::Vec3& vertex) {                  // MxCone.hpp:31-37
    MxShape s; mx::check(mxg_shape_cone(angle, axis.data(), vertex.data(), &s.h_)); return s;
  }
  static MxShape intersection(std::initializer_list<const MxShape*> parts) {                 // MxShapeIntersection.hpp:120-136
    const std::vector<const mxg_shape*> p = raw(parts);
    MxShape s; mx::check(mxg_shape_intersection(p.data(), int(p.size()), &s.h_)); return s;
  }
  static MxShape unite(std::initializer_list<const MxShape*> parts) {                        // MxShapeUnion.hpp:62-78
    const std::vector<const mxg_shape*> p = raw(parts);
    MxShape s; mx::check(mxg_shape_union(p.data(), int(p.size()), &s.h_)); return s;
  }
  static MxShape subtract(const MxShape& base, std::initializer_list<const MxShape*> removed) {   // MxShapeSubtract.hpp:69-92
    const std::vector<const mxg_shape*> p = raw(removed);
    MxShape s; mx::check(mxg_shape_subtract(base.h_, p.data(), int(p.size()), &s.h_)); return s;
  }
  static MxShape mirror(const MxShape& shape, const mx::Vec3& normal, const mx::Vec3& pointInPlane) {    // MxShapeMirror.hpp:85-116
    MxShape s; mx::check(mxg_shape_mirror(shape.h_, normal.data(), pointInPlane.data(), &s.h_)); return s;
  }
  static MxShape repeat(const MxShape& shape, const mx::Vec3& origin, const mx::Vec3& direction, double step, int numPos, int numNeg) {
    MxShape s; mx::check(mxg_shape_repeat(shape.h_, origin.data(), direction.data(), step, numPos, numNeg, &s.h_)); return s;   // MxShapeRepeat.hpp:84-118
  }

  // placement (MxShape.cpp:89-210)
  MxShape& translate(const mx::Vec3& v) { mx::check(mxg_shape_translate(h_, v.data())); return *this; }
  MxShape& rotate(const mx::Vec3& axis, double angle) { mx::check(mxg_shape_rotate(h_, axis.data(), angle, nullptr)); return *this; }
  MxShape& rotate(const mx::Vec3& axis, double angle, const mx::Vec3& pivot) { mx::check(mxg_shape_rotate(h_, axis.data(), angle, pivot.data())); return *this; }
  MxShape& scale(const mx::Vec3& magnitudes, const mx::Vec3& origin = mx::Vec3{{0, 0, 0}}) { mx::check(mxg_shape_scale(h_, magnitudes.data(), origin.data())); return *this; }
  MxShape& reflect(const mx::Vec3& normal, const mx::Vec3& pointInPlane) { mx::check(mxg_shape_reflect(h_, normal.data(), pointInPlane.data())); return *this; }
  MxShape& invert() { mx::check(mxg_shape_invert(h_)); return *this; }

  double func(const mx::Vec3& p) const { double f = 0; mx::check(mxg_shape_eval(h_, p.data(), &f, nullptr)); return f; }   // MxShape.hpp:143-165
  mx::Vec3 gradFunc(const mx::Vec3& p) const { mx::Vec3 g{{0, 0, 0}}; mx::check(mxg_shape_eval(h_, p.data(), nullptr, g.data())); return g; }
  const mxg_shape* raw() const { return h_; }

 private:
  static std::vector<const mxg_shape*> raw(std::initializer_list<const MxShape*> parts) {
    std::vector<const mxg_shape*> v;
    for (const MxShape* s : parts) v.push_back(s ? s->h_ : nullptr);
    return v;
  }
  mxg_shape* h_ = nullptr;
};

class MxEMSim;

// CRS matrix assembled on the device (local column indices, reference entry order). fillComplete<Scalar>() turns the
// rows a map owns into the MxCrsMatrix the eigensolve applies.
class MxDeviceCrs {
 public:
  MxDeviceCrs() = default;
  explicit MxDeviceCrs(mxg_dcsr* h, std::shared_ptr<MxComm> comm) : h_(h), comm_(std::move(comm)) {}
  ~MxDeviceCrs() { if (h_) mxg_dcsr_destroy(h_); }
  MxDeviceCrs(MxDeviceCrs&& o) noexcept : h_(o.h_), comm_(std::move(o.comm_)) { o.h_ = nullptr; }
  MxDeviceCrs& operator=(MxDeviceCrs&& o) noexcept {
    if (this != &o) { if (h_) mxg_dcsr_destroy(h_); h_ = o.h_; comm_ = std::move(o.comm_); o.h_ = nullptr; }
    return *this;
  }
  MxDeviceCrs(const MxDeviceCrs&) = delete;
  MxDeviceCrs& operator=(const MxDeviceCrs&) = delete;

  int64_t numRows() const { return shape()[0]; }
  int64_t numCols() const { return shape()[1]; }
  int64_t numEntries() const { return shape()[2]; }
  bool isComplex() const { return shape()[3] != 0; }

  MxDeviceCrs multiply(const MxDeviceCrs& b) const {                                  // MxCrsMatrix.cpp:358-382
    mxg_dcsr* o = nullptr; mx::check(mxg_dcsr_multiply(h_, b.h_, &o)); return MxDeviceCrs(o, comm_);
  }
  MxDeviceCrs add(MxComplex sa, const MxDeviceCrs& b, MxComplex sb, bool purge = false) const {   // MxCrsMatrix.cpp:401-430
    const double a2[2] = {sa.real(), sa.imag()}, b2[2] = {sb.real(), sb.imag()};
    mxg_dcsr* o = nullptr; mx::check(mxg_dcsr_add(h_, a2, b.h_, b2, purge ? 1 : 0, &o)); return MxDeviceCrs(o, comm_);
  }
  MxDeviceCrs purgeZeros() const { mxg_dcsr* o = nullptr; mx::check(mxg_dcsr_purge(h_, &o)); return MxDeviceCrs(o, comm_); }   // :84-117
  MxDeviceCrs transpose() const { mxg_dcsr* o = nullptr; mx::check(mxg_dcsr_transpose(h_, &o)); return MxDeviceCrs(o, comm_); }
  void scale(MxComplex s) { const double s2[2] = {s.real(), s.imag()}; mx::check(mxg_dcsr_scale(h_, s2)); }

  // MxCrsMatrix::fillComplete (MxCrsMatrix.cpp:325-342): the rows rowMap owns, laid out on the device
  template <class Scalar>
  std::shared_ptr<MxCrsMatrix<Scalar>> fillComplete(std::shared_ptr<MxMap> rowMap, std::shared_ptr<MxMap> domainMap, int layout = 0) const {
    if (mx::ScalarTraits<Scalar>::isComplex != isComplex()) throw std::runtime_error("MxDeviceCrs::fillComplete: scalar type mismatch");
    mxg_crs* A = nullptr;
    mx::check(mxg_crs_create_from_dcsr(rowMap->raw(), domainMap->raw(), h_, layout, &A));
    return std::make_shared<MxCrsMatrix<Scalar>>(A, rowMap, domainMap, true);
  }
  const mxg_dcsr* raw() const { return h_; }

 private:
  std::array<int64_t, 6> shape() const { std::array<int64_t, 6> s{}; mx::check(mxg_dcsr_shape(h_, s.data())); return s; }
  mxg_dcsr* h_ = nullptr;
  std::shared_ptr<MxComm> comm_;
};

// MxEMSim (MxEMSim.cpp:54-199): grid, boundary conditions, PEC shape, dielectric objects; DOF maps and named operators.
class MxEMSim {
 public:
  enum BCType { PERIODIC = 0, ZERO = 1, CONSTANT = 2, PEC = 3, PMC = 4 };

  MxEMSim(std::shared_ptr<MxComm> comm, const std::array<int, 3>& n, const mx::Vec3& origin, const mx::Vec3& size,
          const std::array<int, 3>& lowerBCs = {{0, 0, 0}}, const std::array<int, 3>& upperBCs = {{0, 0, 0}},
          const mx::Vec3& phaseShifts = mx::Vec3{{0, 0, 0}}, double dmFrac = 0.0)
      : comm_(std::move(comm)) {
    mx::check(mxg_sim_create(comm_->raw(), n.data(), origin.data(), size.data(), lowerBCs.data(), upperBCs.data(), phaseShifts.data(), dmFrac, 0, &h_));
    complex_ = phaseShifts[0] != 0 || phaseShifts[1] != 0 || phaseShifts[2] != 0;
  }
  ~MxEMSim() { if (h_) mxg_sim_destroy(h_); }
  MxEMSim(const MxEMSim&) = delete;
  MxEMSim& operator=(const MxEMSim&) = delete;

  void setPEC(const MxShape& shape) { mx::check(mxg_sim_set_pec_shape(h_, shape.raw())); }                       // MxEMSim.cpp:122-129
  void setPECFractions(const std::string& field, const std::vector<double>& fracs) { mx::check(mxg_sim_set_pec_fractions(h_, field.c_str(), fracs.data())); }
  void addDielectric(const MxShape& shape, const std::array<MxComplex, 9>& eps) {                             // MxEMSim.cpp:134-148
    mx::check(mxg_sim_add_dielectric(h_, shape.raw(), reinterpret_cast<const double*>(eps.data())));
    for (const MxComplex& e : eps) complex_ = complex_ || e.imag() != 0;
  }
  void setup() { mx::check(mxg_sim_setup(h_)); }

  // this rank's rows [begin, end) of a field's map (end = -1: to the end); "bfield", "efield", "psifield"
  std::shared_ptr<MxMap> getMap(const std::string& field, int64_t begin = 0, int64_t end = -1) const {
    mxg_map* m = nullptr;
    mx::check(mxg_sim_make_map(h_, field.c_str(), begin, end, &m));
    return std::make_shared<MxMap>(m, comm_, true);
  }
  std::vector<MxIndex> getGlobalIndices(const std::string& field) const {
    int64_t n = 0;
    mx::check(mxg_sim_map_size(h_, field.c_str(), &n, nullptr));
    std::vector<MxIndex> g(static_cast<size_t>(n), 0);
    mx::check(mxg_sim_map_copy(h_, field.c_str(), g.data()));
    return g;
  }
  // MxEMSim::getOp / MxMagWaveOp::initMatrices (MxMagWaveOp.cpp:137-245): curlE curlB divB gradPsi dmA dmL dmVInv mRhs
  // invEps invEpsVolAve curlCurl gradDiv vecLapl scaLapl
  MxDeviceCrs getOp(const std::string& name) const { return getOp(name, complex_); }
  MxDeviceCrs getOp(const std::string& name, bool isComplex) const {
    mxg_dcsr* o = nullptr;
    mx::check(mxg_sim_op(h_, name.c_str(), isComplex ? 1 : 0, nullptr, nullptr, &o));
    return MxDeviceCrs(o, comm_);
  }
  // MxGridFieldInterpolator (MxGridFieldInterpolator.cpp:28-122): `field` of the coarser simulation at this one's DOFs.
  // bloch: Bloch factors across periodic faces (MXG_INTERP_BLOCH, DESIGN.md GMG-bloch).
  MxDeviceCrs interpolatorFrom(const MxEMSim& coarse, const std::string& field, bool bloch = false) const {
    mxg_dcsr* o = nullptr;
    mx::check(mxg_sim_interpolator_ex(coarse.h_, h_, field.c_str(), complex_ ? 1 : 0, bloch ? MXG_INTERP_BLOCH : 0, &o));
    return MxDeviceCrs(o, comm_);
  }
  bool isComplex() const { return complex_; }
  mxg_sim* raw() const { return h_; }

 private:
  std::shared_ptr<MxComm> comm_;
  mxg_sim* h_ = nullptr;
  bool complex_ = false;
};
