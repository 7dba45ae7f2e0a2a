/* mxasm.h -- operator assembly on the device (libmxgpu.so): SURVEY 8 rows f2 (operator generation and the CRS
 * product / sum chains) and f3 (Dey-Mittra cut-cell fractions), the callers that FEED the eigensolve hot path.
 *
 * What it replaces in bauerca/maxwell (paths relative to src/):
 *   MxShape and subclasses (MxCylinder.hpp, MxSphere.hpp, MxHalfSpace.hpp, MxSlab.hpp, MxEllipsoid.hpp, MxTorus.hpp,
 *     MxCone.hpp, MxShapeIntersection.hpp, MxShapeUnion.hpp, MxShapeSubtract.hpp, MxShapeMirror.hpp, MxShapeRepeat.hpp)
 *                                              -> mxg_shape_*
 *   MxEMSim (MxEMSim.cpp:54-199), MxGridField::addShapeRep (MxGridField.cpp:193-226), ::setMap (:256-297)
 *                                              -> mxg_sim_create / _set_pec_shape / _set_pec_fractions / _setup
 *   MxYeeDeyMittraCurlE/CurlB/DivB/GradPsi/Fracs::setMatrix (MxYeeDeyMittraCurlE.cpp:117-178, CurlB.cpp:113-169,
 *     DivB.cpp:157-200, GradPsi.cpp:23-84, Fracs.cpp:30-131), MxMagWaveOp::initMatrices (MxMagWaveOp.cpp:137-245)
 *                                              -> mxg_sim_op
 *   MxCrsMatrix multiply / add / purge (MxCrsMatrix.cpp:84-117,358-430; EpetraExt::MatrixMatrix)
 *                                              -> mxg_dcsr_multiply / _add / _purge / _scale
 *   MxCrsMatrix::fillComplete on the result    -> mxg_crs_create_from_dcsr
 *
 * Results are bit-identical to the reference's host path as restated by the oracle: same entry order inside a row
 * (ascending local column), same order of the floating-point sums, no fused multiply-add, complex quotients as
 * libgcc's __divdc3 forms them. mxg_dcsr_upload brings a host-generated factor into the same algebra.
 *
 * Conventions as in mxgpu.h: plain C, opaque handles, int return codes (0 = ok), message via mxg_last_error(),
 * one host thread per context. Fields are named "bfield", "efield", "psifield". Boundary codes: 0 periodic, 1 zero,
 * 2 constant, 3 PEC wall, 4 PMC wall (MxGridField.h BCType + the PEC/PMC translation of the Yee field classes).
 */
#ifndef MXASM_H
#define MXASM_H

#include <stdint.h>

#include "mxgpu.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mxg_shape mxg_shape; /* CSG solid, host side; f > 0 inside */
typedef struct mxg_sim mxg_sim;     /* grid + boundary conditions + fractions + DOF maps, device resident */
typedef struct mxg_dcsr mxg_dcsr;   /* CRS matrix on the device, local column indices */

/* ---- shapes. Composites copy their parts: parts may be destroyed or moved afterwards. ---- */
int mxg_shape_cylinder(double radius, const double axis[3], const double loc[3], mxg_shape** out);       /* MxCylinder.hpp:34-40 */
int mxg_shape_sphere(double radius, const double loc[3], mxg_shape** out);                               /* MxSphere.hpp:31-33 */
int mxg_shape_halfspace(const double point_in_plane[3], const double normal[3], mxg_shape** out);        /* MxHalfSpace.hpp:31-33 */
int mxg_shape_slab(double thickness, const double normal[3], const double loc[3], mxg_shape** out);      /* MxSlab.hpp:33-39 */
int mxg_shape_ellipsoid(const double loc[3], const double axes[3], mxg_shape** out);                     /* MxEllipsoid.hpp:31-33 */
int mxg_shape_torus(double major_radius, double minor_radius, const double axis[3], const double loc[3], mxg_shape** out); /* MxTorus.hpp:31-37 */
int mxg_shape_cone(double angle, const double axis[3], const double vertex[3], mxg_shape** out);         /* MxCone.hpp:31-37 */
int mxg_shape_intersection(const mxg_shape* const* parts, int n, mxg_shape** out);                       /* MxShapeIntersection.hpp:120-136 */
int mxg_shape_union(const mxg_shape* const* parts, int n, mxg_shape** out);                              /* MxShapeUnion.hpp:62-78 */
int mxg_shape_subtract(const mxg_shape* base, const mxg_shape* const* removed, int n, mxg_shape** out);  /* MxShapeSubtract.hpp:69-92 */
int mxg_shape_mirror(const mxg_shape* shape, const double normal[3], const double point_in_plane[3], mxg_shape** out); /* MxShapeMirror.hpp:85-116 */
int mxg_shape_repeat(const mxg_shape* shape, const double origin[3], const double direction[3], double step, int num_pos,
                     int num_neg, mxg_shape** out);                                                      /* MxShapeRepeat.hpp:84-118 */
int mxg_shape_translate(mxg_shape* s, const double v[3]);                                                /* MxShape.cpp:179-185 */
int mxg_shape_rotate(mxg_shape* s, const double axis[3], double angle, const double* pivot /* NULL: own location */); /* MxShape.cpp:89-125 */
int mxg_shape_scale(mxg_shape* s, const double magnitudes[3], const double origin[3]);                   /* MxShape.cpp:158-168 */
int mxg_shape_reflect(mxg_shape* s, const double normal[3], const double point_in_plane[3]);             /* MxShape.cpp:196-210 */
int mxg_shape_invert(mxg_shape* s);
/* host evaluation: f and/or grad may be NULL (MxShape.hpp:143-165) */
int mxg_shape_eval(const mxg_shape* s, const double p[3], double* f, double grad[3]);
int mxg_shape_destroy(mxg_shape* s);

/* ---- simulation set-up ---- */
/* MxEMSim.cpp:54-120. n cells per direction, lower/upper boundary codes (NULL = periodic), Bloch phase shifts
 * (NULL = 0; non-zero shifts make operators complex by default), Dey-Mittra area-fraction cut-off (MxYeeFitBField). */
int mxg_sim_create(mxg_ctx* ctx, const int n[3], const double origin[3], const double size[3], const int lower[3],
                   const int upper[3], const double phase_shifts[3], double dm_frac, int literal_upper_periodic_e, mxg_sim** out);
int mxg_sim_destroy(mxg_sim* sim); /* destroy the mxg_dcsr matrices made from a simulation before the simulation itself */
/* PEC region from a shape: edge / face / cell fractions of the three fields computed on the device (MxGridField.cpp:193-226) */
int mxg_sim_set_pec_shape(mxg_sim* sim, const mxg_shape* shape);
/* ... or handed in from a host MxGridField: (n0+3)(n1+3)(n2+3) cells of the guarded block x components, cell-major
 * (fields bfield, efield, psifield; dfield as well when dielectrics are present) */
int mxg_sim_set_pec_fractions(mxg_sim* sim, const char* field, const double* fracs);
/* MxEMSim::addDielectric (MxEMSim.cpp:134-148): a shape filled with the permittivity tensor eps (3x3 complex, row-major
 * (re, im) pairs; up to 4 objects). Its edge / dual-face / cell fractions are computed on the device; the operators
 * "invEps" (MxYeeFitInvEps.cpp:420-596) and "invEpsVolAve" (:650-725) become available and the chains use them. */
int mxg_sim_add_dielectric(mxg_sim* sim, const mxg_shape* shape, const double eps[18]);
int mxg_sim_setup(mxg_sim* sim); /* DOF maps of B, E and psi (MxGridField.cpp:256-297 with the Dey-Mittra overrides) */
int mxg_sim_map_size(mxg_sim* sim, const char* field, int64_t* num_local, int64_t* num_global);
int mxg_sim_map_copy(mxg_sim* sim, const char* field, int64_t* gids);
int mxg_sim_fractions(mxg_sim* sim, const char* field, double* out); /* guarded-block layout as above */
/* rows [begin, end) of a field's map as an mxg_map of the context (end = -1: to the end) */
int mxg_sim_make_map(mxg_sim* sim, const char* field, int64_t begin, int64_t end, mxg_map** out);

/* ---- operators ---- */
/* name: curlE curlB divB gradPsi dmA dmL dmVInv mRhs invEps invEpsVolAve curlCurl gradDiv vecLapl scaLapl
 * (MxEMOps.cpp:39-168, MxMagWaveOp.cpp:137-245). inv_eps / inv_eps_vol_ave: optional replacements for the dielectric
 * factors of the chains (NULL: generated from the simulation's dielectric objects, identity without any). */
int mxg_sim_op(mxg_sim* sim, const char* name, int is_complex, const mxg_dcsr* inv_eps, const mxg_dcsr* inv_eps_vol_ave,
               mxg_dcsr** out);
/* The rows [row_begin, row_end) (positions in the row field's map) of mxg_sim_op's operator, bit for bit, assembled from
 * the rows the chain needs only: each factor on the rows the factor to its left references (an x-slab +- the stencil
 * reach, wrapping around on periodic-x grids), multiplied in the reference's association order (MxMagWaveOp.cpp:137-245,
 * MxEMOps.cpp:39-168). inv_eps / inv_eps_vol_ave may be whole or partial; they must store the rows the chain needs.
 * Out-of-range or inverted ranges return an error code. */
int mxg_sim_op_rows(mxg_sim* sim, const char* name, int is_complex, const mxg_dcsr* inv_eps, const mxg_dcsr* inv_eps_vol_ave,
                    int64_t row_begin, int64_t row_end, mxg_dcsr** out);
int mxg_dcsr_upload(mxg_sim* sim, const char* row_field, const char* col_field, int64_t nrows, int64_t ncols,
                    const int64_t* rowptr, const int32_t* col, const double* vals, int is_complex, mxg_dcsr** out);
/* A matrix may store only some rows of its map (mxg_dcsr_rows). multiply: rows of a x b on a's stored rows; b must store
 * every row a's columns reference, otherwise an error ("a column of A has no stored row in B"). add: b must store a's rows. */
int mxg_dcsr_multiply(const mxg_dcsr* a, const mxg_dcsr* b, mxg_dcsr** out);                     /* MxCrsMatrix.cpp:358-382 */
int mxg_dcsr_add(const mxg_dcsr* a, const double sa[2], const mxg_dcsr* b, const double sb[2], int purge, mxg_dcsr** out); /* :401-430 */
int mxg_dcsr_purge(const mxg_dcsr* a, mxg_dcsr** out);                                           /* MxCrsMatrix.cpp:84-117 */
int mxg_dcsr_scale(mxg_dcsr* a, const double s[2]);
/* conjugate transpose, rows sorted by column; a must store all its rows (the rows of a restriction:
 * mxg_sim_interpolator_transpose_rows) */
int mxg_dcsr_transpose(const mxg_dcsr* a, mxg_dcsr** out);
/* MxGridFieldInterpolator (MxGridFieldInterpolator.cpp:28-122): `field` of sim_from interpolated at the DOFs of sim_to --
 * the refiners / coarseners of MxGeoMultigridPrec (MxGeoMultigridPrec.cpp:98-240). Rows on sim_to, columns on sim_from. */
int mxg_sim_interpolator(mxg_sim* sim_from, mxg_sim* sim_to, const char* field, int is_complex, mxg_dcsr** out);
/* rows [row_begin, row_end) of sim_to's map of the same interpolator (MxGridFieldInterpolator.cpp:28-122) */
int mxg_sim_interpolator_rows(mxg_sim* sim_from, mxg_sim* sim_to, const char* field, int is_complex,
                              int64_t row_begin, int64_t row_end, mxg_dcsr** out);
/* rows [row_begin, row_end) of sim_from's map of its conjugate transpose (the restriction of MxGeoMultigridPrec.cpp:98-240
 * before the 1/8 scaling): the interpolator is generated on the fine rows that can reach those coarse rows only */
int mxg_sim_interpolator_transpose_rows(mxg_sim* sim_from, mxg_sim* sim_to, const char* field, int is_complex,
                                        int64_t row_begin, int64_t row_end, mxg_dcsr** out);
/* The same three with flags (the plain ones are flags = 0). MXG_INTERP_BLOCH: a stencil cell that wraps across a periodic
 * face of sim_from carries that direction's Bloch factor, e^{+i phi} from the top and e^{-i phi} from below, so that the
 * prolongator maps a coarse Bloch-periodic field onto the fine one (MxGridFieldInterpolator.cpp:28-122 applies none;
 * DESIGN.md deviation GMG-bloch). Both simulations must have the same phase shifts; a real (is_complex = 0) transfer with
 * a non-zero phase is an error; with all phases 0 the result equals the plain transfer bit for bit. */
#define MXG_INTERP_BLOCH 1
int mxg_sim_interpolator_ex(mxg_sim* sim_from, mxg_sim* sim_to, const char* field, int is_complex, int flags, mxg_dcsr** out);
int mxg_sim_interpolator_rows_ex(mxg_sim* sim_from, mxg_sim* sim_to, const char* field, int is_complex,
                                 int64_t row_begin, int64_t row_end, int flags, mxg_dcsr** out);
int mxg_sim_interpolator_transpose_rows_ex(mxg_sim* sim_from, mxg_sim* sim_to, const char* field, int is_complex,
                                           int64_t row_begin, int64_t row_end, int flags, mxg_dcsr** out);
/* out = {rows, columns, entries, is_complex, row field, column field}; fields 0 B, 1 E, 2 psi, -1 unknown. rows counts
 * the stored rows. */
int mxg_dcsr_shape(const mxg_dcsr* a, int64_t out[6]);
/* out = {first, end}: map positions of the stored rows (0 and the map size for a whole-map matrix) */
int mxg_dcsr_rows(const mxg_dcsr* a, int64_t out[2]);
/* stored rows [row_begin, row_end) to the host; rowptr is rebased to 0; col / vals may be NULL */
int mxg_dcsr_download(const mxg_dcsr* a, int64_t row_begin, int64_t row_end, int64_t* rowptr, int32_t* col, double* vals);
int mxg_dcsr_destroy(mxg_dcsr* a);

/* MxCrsMatrix::fillComplete (MxCrsMatrix.cpp:325-342) for a device-assembled operator: the rows row_map owns become an
 * mxg_crs (layout: MXG_LAYOUT_* of mxgpu.h, 0 = default). Collective when the context has several ranks. */
int mxg_crs_create_from_dcsr(mxg_map* row_map, mxg_map* domain_map, const mxg_dcsr* a, int layout, mxg_crs** out);

/* Device bytes held by the assembly of a context's simulations (fractions, maps, matrices, temporaries):
 * out = {current, peak}; reset_peak != 0 restarts the peak at the current value. */
int mxg_asm_memory(mxg_ctx* ctx, int64_t out[2], int reset_peak);

#ifdef __cplusplus
}
#endif
#endif
