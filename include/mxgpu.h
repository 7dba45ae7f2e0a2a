/* libmxgpu -- C ABI of the B200 (sm_100a) eigensolve inner loop for bauerca/maxwell.
 *
 * This is the drop-in boundary: every entry point replaces one call the reference makes
 * into Epetra through its MxMap / MxMultiVector / MxAnasaziMV / MxCrsMatrix wrappers
 * (file:line cited per function, paths relative to the reference's src/). Plain pointers
 * and sizes only; no C++ or torch types cross this interface.
 *
 * Conventions
 *  - One process drives one GPU (one "rank"). Multi-GPU = one process per GPU; ranks are
 *    wired together with mxg_ctx_comm_init (NCCL over NVLink), replacing MxComm/Epetra_MpiComm.
 *  - Every function returns 0 on success and a negative code on failure; the message is
 *    available from mxg_last_error() (the reference prints and exit()s / throws 1 instead,
 *    e.g. MxAnasaziMV.cpp:20-23, MxCrsMatrix.cpp:89-91 -- the C++ shims turn non-zero
 *    into std::runtime_error).
 *  - Scalars are passed as double[2] = {re, im}; im is ignored for real objects.
 *  - Multivectors are column-major, local stride = local length. Complex entries are
 *    interleaved (re, im), bit-compatible with std::complex<double> and with the
 *    reference's 2N real storage (MxMap.cpp:90-108, MxMultiVector.hpp:119-130).
 *  - Host dense matrices (Teuchos::SerialDenseMatrix in the reference) are column-major
 *    with leading dimension ld, complex interleaved.
 *  - All calls on one ctx must come from one host thread. Calls are asynchronous on the
 *    ctx stream; only the reducing / downloading calls synchronise.
 *  - There is no CPU fallback: without a CUDA device mxg_ctx_create fails.
 */
#ifndef MXGPU_H
#define MXGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mxg_ctx mxg_ctx;
typedef struct mxg_map mxg_map;
typedef struct mxg_mv mxg_mv;
typedef struct mxg_crs mxg_crs;

#define MXG_OK 0
#define MXG_ERR_CUDA -1
#define MXG_ERR_ARG -2
#define MXG_ERR_NCCL -3
#define MXG_ERR_STATE -4

#define MXG_MAX_COLS 128      /* widest multivector / view a single call accepts */
#define MXG_UNIQUE_ID_BYTES 128

const char* mxg_last_error(void);
int mxg_version(void);

/* ---- context and communicator (replaces MxComm, MxComm.hpp:14-37) ---------------------- */
int mxg_ctx_create(int device, mxg_ctx** out);
int mxg_ctx_destroy(mxg_ctx* ctx);
int mxg_ctx_sync(mxg_ctx* ctx);
int mxg_ctx_rank(const mxg_ctx* ctx);        /* MxComm::myPID  */
int mxg_ctx_num_ranks(const mxg_ctx* ctx);   /* MxComm::numProc */
/* NCCL wiring: rank 0 calls mxg_comm_unique_id and ships the bytes to the other ranks by
 * any means (the tests use torch.distributed); then every rank calls mxg_ctx_comm_init. */
int mxg_comm_unique_id(void* out /* MXG_UNIQUE_ID_BYTES */);
int mxg_ctx_comm_init(mxg_ctx* ctx, int rank, int nranks, const void* unique_id);
/* Counter that advances on every call: MxMultiVector::random() mixes it into its seed so that successive MvRandom calls --
 * also on Clone()d blocks -- draw independent numbers, as Epetra's Random() does by advancing its state
 * (MxMultiVector.hpp:41). Ranks that make the same calls see the same values, which keeps vectors rank-count invariant. */
uint64_t mxg_ctx_random_epoch(mxg_ctx* ctx);
/* raw handles for host code that wants to enqueue its own work or events */
void* mxg_ctx_stream(mxg_ctx* ctx);          /* cudaStream_t */
/* device timing on the ctx stream (CUDA events; slot in 0..15). The reference times with
 * Epetra_Time wall clocks (MxSolver.cpp:102,111; MxMagWaveOp.cpp:96-115). */
int mxg_ctx_event_record(mxg_ctx* ctx, int slot);
int mxg_ctx_event_elapsed_ms(mxg_ctx* ctx, int slot_begin, int slot_end, double* ms);
/* pinned host buffers for callers that stream vectors through upload/download */
void* mxg_host_alloc(size_t bytes);
void mxg_host_free(void* p);

/* ---- maps (MxMap.hpp:22-103, MxMap.cpp:60-81) ------------------------------------------
 * A map is this rank's list of owned global DOF ids. GIDs must be ascending within a rank
 * and rank r's GIDs must all precede rank r+1's (x-slab partition; see DESIGN.md). */
int mxg_map_create(mxg_ctx* ctx, int64_t n_global, const int64_t* my_gids, int64_t n_local, mxg_map** out);
/* Same map with a component-major DEVICE ordering of the multivectors that live on it (component = GID mod ncomp, the
 * reference's globCompIndx = comp + ncomp * cell, MxGridField.hpp:142-145): consecutive device positions are
 * consecutive cells of one field component, which makes the gathers of the curl-curl SpMM contiguous. Single-rank
 * contexts only. mxg_mv_upload / mxg_mv_download / mxg_mv_col_ptr then use device order; mxg_map_get_order returns
 * perm[device position] = reference local index so callers can translate (returns 1 if ordered, 0 if identity).
 * Everything else (block operations, mxg_crs_create, mxg_mv_random, mxg_mv_to_grid) is order-agnostic. */
int mxg_map_create_ordered(mxg_ctx* ctx, int64_t n_global, const int64_t* my_gids, int64_t n_local, int ncomp, mxg_map** out);
int mxg_map_get_order(const mxg_map* map, int32_t* perm_out);
int mxg_map_destroy(mxg_map* map);
int64_t mxg_map_local_size(const mxg_map* map);    /* getNodeNumIndices   */
int64_t mxg_map_global_size(const mxg_map* map);   /* getGlobalNumIndices */

/* ---- multivectors (MxMultiVector.hpp:16-89, MxAnasaziMV.hpp:23-136) -------------------- */
/* MxMultiVector(map, numVecs) / MxAnasaziMV::Clone: zero-initialised n x ncols block */
int mxg_mv_create(mxg_map* map, int ncols, int is_complex, mxg_mv** out);
/* CloneCopy() (cols == NULL) / CloneCopy(index): deep copy of the listed columns */
int mxg_mv_clone_copy(const mxg_mv* src, const int* cols, int ncols, mxg_mv** out);
/* CloneView / CloneViewNonConst (MxMultiVector.cpp:29-44): shares storage with the parent;
 * arbitrary column lists are legal; the parent allocation lives until the last view dies */
int mxg_mv_view(mxg_mv* parent, const int* cols, int ncols, mxg_mv** out);
int mxg_mv_destroy(mxg_mv* mv);
int mxg_mv_num_cols(const mxg_mv* mv);              /* GetNumberVecs */
int64_t mxg_mv_local_length(const mxg_mv* mv);      /* getLocalLength (complex count) */
int64_t mxg_mv_global_length(const mxg_mv* mv);     /* GetVecLength, MxAnasaziMV.hpp:77-79 */
int mxg_mv_is_complex(const mxg_mv* mv);
/* SetBlock (MxAnasaziMV.cpp:201-213): column index[j] of dst = column j of src */
int mxg_mv_set_block(mxg_mv* dst, const mxg_mv* src, const int* index, int n);
/* operator= (MxMultiVector.cpp:62-82): same shape, deep copy */
int mxg_mv_assign(mxg_mv* dst, const mxg_mv* src);
/* set / MvInit (MxMultiVector.cpp:86-91, MxAnasaziMV.hpp:125-132) */
int mxg_mv_fill(mxg_mv* mv, const double alpha[2]);
/* random / MvRandom (MxMultiVector.hpp:41): uniform (-1,1) keyed by (seed, global DOF id,
 * column position in the underlying allocation) so the result is independent of the GPU count */
int mxg_mv_random(mxg_mv* mv, uint64_t seed);
/* scale(Scalar) / MvScale(alpha) (MxMultiVector.cpp:97-113) */
int mxg_mv_scale(mxg_mv* mv, const double alpha[2]);
/* scale(vector) / MvScale(vector) (MxMultiVector.cpp:116-123); alphas: ncols scalars */
int mxg_mv_scale_cols(mxg_mv* mv, const double* alphas);
/* conj (MxMultiVector.cpp:128-140) */
int mxg_mv_conj(mxg_mv* mv);
/* update: dst = a*A + s*dst (MxMultiVector.cpp:205-227) */
int mxg_mv_update(mxg_mv* dst, const double a[2], const mxg_mv* A, const double s[2]);
/* MvAddMv: dst = alpha*A + beta*B; A and/or B may alias dst (MxAnasaziMV.cpp:89-111) */
int mxg_mv_add_mv(mxg_mv* dst, const double alpha[2], const mxg_mv* A, const double beta[2], const mxg_mv* B);
/* dst_j = alphas[j]*A_j + betas[j]*B_j: MvAddMv with one scalar pair per column (as MvScale(vector), MxAnasaziMV.hpp:110-118,
 * followed by MvAddMv, MxAnasaziMV.cpp:89-111, in one pass); alphas/betas: ncols scalars; A and/or B may alias dst */
int mxg_mv_axpby_cols(mxg_mv* dst, const double* alphas, const mxg_mv* A, const double* betas, const mxg_mv* B);
/* removeConstField (MxGeoMultigridPrec.cpp:400-411, MxUtil.cpp:483-503): x_j -= (x_j . 1)/(1 . 1) 1 for every column;
 * reduction, all-reduce and update run back to back on the device */
int mxg_mv_remove_const_field(mxg_mv* mv);
/* MxGridField::zeroUnusedComponents (MxGridField.cpp:548-576; applied to the initial block at MxSolver.cpp:65):
 * zero the entries whose shape fraction is 0; fracs = one-column multivector on the same map */
int mxg_mv_zero_unused(mxg_mv* mv, const mxg_mv* fracs);
/* norm2 / MvNorm (MxMultiVector.cpp:148-155): out[ncols] */
int mxg_mv_norm2(const mxg_mv* mv, double* out);
/* dot / MvDot: out[j] = conj(a_j) . b_j  (out: ncols scalars, complex interleaved). This is
 * the mathematical inner product; the reference's complex version returns Im = 0
 * (MxMultiVector.cpp:186-203, see DESIGN.md R12). */
int mxg_mv_dot(const mxg_mv* a, const mxg_mv* b, double* out);
/* normalize() as intended (divide each column by its 2-norm); the reference multiplies
 * (MxMultiVector.cpp:157-172, DESIGN.md R12) */
int mxg_mv_normalize(mxg_mv* mv);
/* MvTransMv: B(k x b, host) = alpha * A^H * X, summed over all ranks
 * (MxAnasaziMV.cpp:114-149 real, :152-197 complex) */
int mxg_mv_trans_mv(const double alpha[2], const mxg_mv* A, const mxg_mv* X, double* B, int ldb);
/* MvTimesMatAddMv: Y = alpha * A * B + beta * Y, B host k x b
 * (MxAnasaziMV.cpp:8-33 real, :40-86 complex) */
int mxg_mv_times_mat_add_mv(const double alpha[2], const mxg_mv* A, const double* B, int ldb,
                            const double beta[2], mxg_mv* Y);
/* host <-> device transfers of the local block (tests, I/O, the e2e bench leg);
 * host layout: column-major, leading dimension ld (in scalars) */
int mxg_mv_upload(mxg_mv* mv, const double* host, int64_t ld);
int mxg_mv_download(const mxg_mv* mv, double* host, int64_t ld);
/* the map a multivector / operator lives on (borrowed handle; getMap(), getRangeMap(), getDomainMap()) */
mxg_map* mxg_mv_get_map(const mxg_mv* mv);
mxg_map* mxg_crs_row_map(const mxg_crs* A);
mxg_map* mxg_crs_domain_map(const mxg_crs* A);
/* Field output in the layout of MxIO::save (MxIO.cpp:166-221): column `col` scattered into a dense array over the
 * GID range [gid_lo, gid_hi) -- GID = comp + numComps * cell, cell z-fastest over the node grid (MxGrid.h:96-114) --
 * with zeros where the map holds no DOF. Host buffers of gid_hi - gid_lo doubles; out_imag only for complex fields.
 * A slab rank passes the GID range of its own planes. */
int mxg_mv_to_grid(const mxg_mv* mv, int col, int64_t gid_lo, int64_t gid_hi, double* out_real, double* out_imag);
/* device pointer of column j (for host code that enqueues its own kernels) */
void* mxg_mv_col_ptr(mxg_mv* mv, int j);

/* ---- sparse operators (MxCrsMatrix.hpp:14-82) -------------------------------------------
 * mxg_crs_create takes the rows this rank owns in host CSR form with GLOBAL column ids --
 * what insertRowValues + fillComplete hand to Epetra (MxCrsMatrix.cpp:122-170,325-342) --
 * and builds the device layout (pattern-compressed sliced ELL, halo plan) inside.
 * rowptr has n_local_rows+1 entries; vals has nnz scalars (complex interleaved).
 * Duplicate (row, col) entries are summed; explicit zeros are kept. */
int mxg_crs_create(mxg_map* row_map, mxg_map* domain_map, const int64_t* rowptr, const int64_t* col_gids,
                   const double* vals, int is_complex, mxg_crs** out);
/* same, with an explicit device layout: 0 = pattern dictionary + sliced ELL (default),
 * 1 = sliced ELL only (every row stored explicitly; the plain-CRS-traffic baseline).
 * mxg_crs_create reads the default from the environment variable MXG_SPMV_LAYOUT=dict|sell. */
int mxg_crs_create_opts(mxg_map* row_map, mxg_map* domain_map, const int64_t* rowptr, const int64_t* col_gids,
                        const double* vals, int is_complex, int layout, mxg_crs** out);
/* On several ranks an operator with a peer-memory halo owns buffers its neighbours have mapped (CUDA IPC): destroy it on every
 * rank at the same point of the program, after a barrier / synchronisation of all ranks (no rank may still be applying it). */
int mxg_crs_destroy(mxg_crs* A);
/* apply (MxCrsMatrix.cpp:347-353): y = A x; x over the domain map, y over the row map.
 * On several ranks the ghost entries of x are exchanged with NCCL send/recv, overlapped
 * with the rows that need no ghosts. x and y must not alias. */
int mxg_crs_apply(const mxg_crs* A, const mxg_mv* x, mxg_mv* y);
/* Host-buffer form of apply for callers that keep their vectors in host memory (what MxCrsMatrix::apply sees when
 * the multivectors are still Epetra objects): y_host[i] = A x_host[i], i < count, one column each, local length of the
 * domain / row map, (re,im) interleaved for complex operators. Uploads, applies and downloads are pipelined over two
 * device slots; pinned host buffers (mxg_host_alloc) make the copies asynchronous. Returns when every y is complete. */
int mxg_crs_apply_host_batch(const mxg_crs* A, int count, const double* const* x_host, double* const* y_host);
/* y = alpha*A*x + beta*y fused into the SpMM epilogue (residuals r = b - A x of the
 * multigrid cycle, MxGeoMultigridPrec.cpp:312-314; shifted operators, MxMagWaveOp.cpp:247-256) */
int mxg_crs_apply_axpby(const mxg_crs* A, const double alpha[2], const mxg_mv* x, const double beta[2], mxg_mv* y);
/* one apply, on the path mxg_crs_apply takes, split into phases. ms[3] = whole apply (CUDA events) on every path.
 * One rank (CUDA events): ms[0] = dictionary-row kernel, ms[1] = sliced-ELL kernel, ms[2] = time before the first kernel.
 * Several ranks, single launch over peer memory (the %globaltimer roles of mxg_crs_trace): ms[0] = interior rows (roles 1
 * and 2, first start to last end), ms[1] = boundary rows (role 4), ms[2] = pack + flag publish (role 0); a role that did
 * not run counts 0.
 * Several ranks, NCCL exchange (CUDA events): ms[0] = interior rows up to the end of the apply, ms[1] = boundary rows,
 * ms[2] = NCCL send/recv. */
int mxg_crs_apply_timed(const mxg_crs* A, const mxg_mv* x, mxg_mv* y, double ms[4]);
/* %globaltimer timeline of ONE multi-rank apply (the single-launch path): call with enable = 1, apply once, call with
 * enable = 0 to read out[10] in ns relative to the earliest mark -- role r: out[2r] first start, out[2r+1] last end;
 * roles: 0 pack + flag publish, 1 interior dictionary rows, 2 interior sliced-ELL rows, 3 boundary blocks waiting for the
 * neighbours' flags, 4 boundary rows. Entries of roles that did not run are -1. */
int mxg_crs_trace(const mxg_crs* A, int enable, double out[10]);
/* layout statistics: out[0]=local rows, [1]=local nnz, [2]=rows on the dictionary path,
 * [3]=distinct row patterns, [4]=device bytes of the matrix layout, [5]=ghost entries,
 * [6]=rows that need ghosts, [7]=padded ELL entries */
int mxg_crs_stats(const mxg_crs* A, int64_t out[8]);
/* y = d .* x with d a one-column multivector: diagonal operators such as mRhs = dmA
 * (MxMagWaveOp.cpp:227-241, applied at :865,895,1132) without a CRS round trip */
int mxg_mv_diag_mult(mxg_mv* y, const mxg_mv* d, const mxg_mv* x);

/* y = diag(A)^-1 x (Jacobi preconditioner of the projection solve; A must be square on one map) */
int mxg_crs_jacobi(const mxg_crs* A, const mxg_mv* x, mxg_mv* y);

/* ---- geometric multigrid preconditioner (MxGeoMultigridPrec.{h,cpp}; dead code in the
 * reference, so this follows its structure: setup :98-240, vCycle :243-398, fullVCycle
 * :547-616, ApplyInverse :496-542). Levels are ordered fine -> coarse. ops[l] must be square
 * on one map; restrictors[l] maps level l -> l+1, prolongators[l] maps level l+1 -> l.
 * The handles are borrowed: they must outlive the preconditioner. ------------------------ */
typedef struct mxg_gmg mxg_gmg;
typedef struct mxg_gmg_params {
  int smoother_degree;      /* Chebyshev degree per smoothing step ("smoother sweeps")      */
  double eig_ratio;         /* smoother targets [lmax/ratio, 1.1*lmax] ("ratio eigenvalue") */
  int cycles;               /* V-cycles per apply ("cycles")                                 */
  int coarse_degree;        /* Chebyshev degree of the coarsest-level solve (replaces KLU)  */
  double coarse_eig_ratio;
  int full_multigrid;       /* 1: fullVCycle (FMG), 0: plain V-cycles from a zero guess     */
  int power_iterations;     /* iterations of the lambda_max(D^-1 A) estimate at setup       */
  int remove_const_field;   /* 1: project the constant out after every coarsen / refine ("remove const field",
                               MxGeoMultigridPrec.cpp:108,438-452): singular scalar Laplacians    */
} mxg_gmg_params;
void mxg_gmg_default_params(mxg_gmg_params* p);
int mxg_gmg_create(mxg_ctx* ctx, int nlevels, mxg_crs* const* ops, mxg_crs* const* restrictors,
                   mxg_crs* const* prolongators, const mxg_gmg_params* params, mxg_gmg** out);
int mxg_gmg_destroy(mxg_gmg* g);
/* ApplyInverse: x = M^-1 b for a block of right-hand sides */
int mxg_gmg_apply(mxg_gmg* g, const mxg_mv* b, mxg_mv* x);
/* out[0]=rows, [1]=nnz, [2]=lambda_max estimate of D^-1 A on that level, [3]=SpMM count so far */
int mxg_gmg_info(const mxg_gmg* g, int level, double out[4]);

/* number of kernels this library has launched on ctx since creation (bench bookkeeping) */
int64_t mxg_ctx_launch_count(const mxg_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* MXGPU_H */
