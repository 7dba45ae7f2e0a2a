"""maxwell_b200 -- B200-native eigensolve inner loop for bauerca/maxwell.

The product is libmxgpu.so (hand-written sm_100a CUDA behind the C ABI in include/mxgpu.h)
plus the C++ shim classes in include/mx/. This Python module is only a ctypes veneer with the
reference's class and method names (MxMap, MxMultiVector / MxAnasaziMV, MxCrsMatrix) so tests
and bench.py read like the reference's own call sites. It never falls back to a CPU path: if
the library is missing or no GPU is present, construction fails loudly.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

MAX_COLS = 128
LAYOUT_DICT, LAYOUT_SELL = 0, 1


class MxError(RuntimeError):
    pass


def library_path():
    return os.path.join(_HERE, "libmxgpu.so")


def load_library():
    """dlopen libmxgpu.so and declare every entry point of include/mxgpu.h."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise MxError("libmxgpu.so not built (run `python __graft_entry__.py`); there is no CPU fallback")
    L = C.CDLL(path, mode=C.RTLD_GLOBAL)
    vp, i64, i32, dp = C.c_void_p, C.c_int64, C.c_int, C.POINTER(C.c_double)
    pvp = C.POINTER(vp)
    ip = C.POINTER(C.c_int)
    sig = {
        "mxg_last_error": (C.c_char_p, []),
        "mxg_version": (i32, []),
        "mxg_ctx_create": (i32, [i32, pvp]),
        "mxg_ctx_destroy": (i32, [vp]),
        "mxg_ctx_sync": (i32, [vp]),
        "mxg_ctx_rank": (i32, [vp]),
        "mxg_ctx_num_ranks": (i32, [vp]),
        "mxg_comm_unique_id": (i32, [vp]),
        "mxg_ctx_comm_init": (i32, [vp, i32, i32, vp]),
        "mxg_ctx_stream": (vp, [vp]),
        "mxg_ctx_launch_count": (i64, [vp]),
        "mxg_ctx_event_record": (i32, [vp, i32]),
        "mxg_ctx_event_elapsed_ms": (i32, [vp, i32, i32, dp]),
        "mxg_host_alloc": (vp, [C.c_size_t]),
        "mxg_host_free": (None, [vp]),
        "mxg_crs_apply_timed": (i32, [vp, vp, vp, dp]),
        "mxg_map_create": (i32, [vp, i64, vp, i64, pvp]),
        "mxg_map_create_ordered": (i32, [vp, i64, vp, i64, i32, pvp]),
        "mxg_map_get_order": (i32, [vp, vp]),
        "mxg_map_destroy": (i32, [vp]),
        "mxg_map_local_size": (i64, [vp]),
        "mxg_map_global_size": (i64, [vp]),
        "mxg_mv_create": (i32, [vp, i32, i32, pvp]),
        "mxg_mv_clone_copy": (i32, [vp, ip, i32, pvp]),
        "mxg_mv_view": (i32, [vp, ip, i32, pvp]),
        "mxg_mv_destroy": (i32, [vp]),
        "mxg_mv_num_cols": (i32, [vp]),
        "mxg_mv_local_length": (i64, [vp]),
        "mxg_mv_global_length": (i64, [vp]),
        "mxg_mv_is_complex": (i32, [vp]),
        "mxg_mv_set_block": (i32, [vp, vp, ip, i32]),
        "mxg_mv_assign": (i32, [vp, vp]),
        "mxg_mv_fill": (i32, [vp, dp]),
        "mxg_mv_random": (i32, [vp, C.c_uint64]),
        "mxg_mv_scale": (i32, [vp, dp]),
        "mxg_mv_scale_cols": (i32, [vp, vp]),
        "mxg_mv_conj": (i32, [vp]),
        "mxg_mv_update": (i32, [vp, dp, vp, dp]),
        "mxg_mv_add_mv": (i32, [vp, dp, vp, dp, vp]),
        "mxg_mv_axpby_cols": (i32, [vp, vp, vp, vp, vp]),
        "mxg_mv_remove_const_field": (i32, [vp]),
        "mxg_mv_zero_unused": (i32, [vp, vp]),
        "mxg_mv_norm2": (i32, [vp, vp]),
        "mxg_mv_dot": (i32, [vp, vp, vp]),
        "mxg_mv_normalize": (i32, [vp]),
        "mxg_mv_trans_mv": (i32, [dp, vp, vp, vp, i32]),
        "mxg_mv_times_mat_add_mv": (i32, [dp, vp, vp, i32, dp, vp]),
        "mxg_mv_upload": (i32, [vp, vp, i64]),
        "mxg_mv_download": (i32, [vp, vp, i64]),
        "mxg_mv_to_grid": (i32, [vp, i32, i64, i64, vp, vp]),
        "mxg_mv_col_ptr": (vp, [vp, i32]),
        "mxg_crs_create": (i32, [vp, vp, vp, vp, vp, i32, pvp]),
        "mxg_crs_create_opts": (i32, [vp, vp, vp, vp, vp, i32, i32, pvp]),
        "mxg_crs_destroy": (i32, [vp]),
        "mxg_crs_apply": (i32, [vp, vp, vp]),
        "mxg_crs_apply_host_batch": (i32, [vp, i32, vp, vp]),
        "mxg_crs_apply_axpby": (i32, [vp, dp, vp, dp, vp]),
        "mxg_crs_stats": (i32, [vp, vp]),
        "mxg_crs_trace": (i32, [vp, i32, vp]),
        "mxg_mv_get_map": (vp, [vp]),
        "mxg_crs_row_map": (vp, [vp]),
        "mxg_crs_domain_map": (vp, [vp]),
        "mxg_mv_diag_mult": (i32, [vp, vp, vp]),
        "mxg_crs_jacobi": (i32, [vp, vp, vp]),
        "mxg_gmg_default_params": (None, [vp]),
        "mxg_gmg_create": (i32, [vp, i32, vp, vp, vp, vp, pvp]),
        "mxg_gmg_destroy": (i32, [vp]),
        "mxg_gmg_apply": (i32, [vp, vp, vp]),
        "mxg_gmg_info": (i32, [vp, i32, dp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _LIB = L
    return L


_SOLVER = None


class GmgParams(C.Structure):
    """mxg_gmg_params (include/mxgpu.h)."""
    _fields_ = [("smoother_degree", C.c_int), ("eig_ratio", C.c_double), ("cycles", C.c_int), ("coarse_degree", C.c_int),
                ("coarse_eig_ratio", C.c_double), ("full_multigrid", C.c_int), ("power_iterations", C.c_int),
                ("remove_const_field", C.c_int)]


class SolverParams(C.Structure):
    """mxs_params (include/mxsolver.h)."""
    _fields_ = [("nev", C.c_int), ("block_size", C.c_int), ("max_iters", C.c_int), ("tol", C.c_double), ("verbose", C.c_int),
                ("seed", C.c_uint64), ("random_init", C.c_int)]


class Projection(C.Structure):
    """mxs_projection (include/mxsolver.h): the divergence-cleaning projection as an eigensolver constraint."""
    _fields_ = [("divB", C.c_void_p), ("gradPsi", C.c_void_p), ("scaLapl", C.c_void_p), ("sca_prec", C.c_void_p),
                ("tol_init", C.c_double), ("tol_w", C.c_double), ("tol_x", C.c_double), ("reproject_ratio", C.c_double),
                ("max_iters", C.c_int), ("max_iters_w", C.c_int)]


def load_solver():
    """dlopen libmxsolver.so (host C++ driver above the C ABI: include/mx/MxSolver.hpp)."""
    global _SOLVER
    if _SOLVER is not None:
        return _SOLVER
    load_library()
    path = os.path.join(_HERE, "libmxsolver.so")
    if not os.path.exists(path):
        raise MxError("libmxsolver.so not built (run `python __graft_entry__.py`)")
    S = C.CDLL(path, mode=C.RTLD_GLOBAL)
    vp, dp = C.c_void_p, C.POINTER(C.c_double)
    S.mxs_default_params.restype = None
    S.mxs_default_params.argtypes = [vp]
    S.mxs_last_error.restype = C.c_char_p
    S.mxs_lobpcg.restype = C.c_int
    S.mxs_lobpcg.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, dp]
    S.mxs_check_eigensolution.restype = C.c_int
    S.mxs_check_eigensolution.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    S.mxs_mag_to_elec.restype = C.c_int
    S.mxs_mag_to_elec.argtypes = [vp, vp, vp, vp, vp]
    S.mxs_eigvals_to_freqs.restype = C.c_int
    S.mxs_eigvals_to_freqs.argtypes = [vp, vp, C.c_int, C.c_double, C.c_int, vp, vp]
    S.mxs_magwave_apply.restype = C.c_int
    S.mxs_magwave_apply.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, C.c_double, C.c_double, C.c_int, vp, vp, vp]
    S.mxs_last_profile.restype = None
    S.mxs_last_profile.argtypes = [vp]
    S.mxs_last_profile_ex.restype = None
    S.mxs_last_profile_ex.argtypes = [vp]
    S.mxs_lobpcg_projected.restype = C.c_int
    S.mxs_lobpcg_projected.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, dp]
    S.mxs_div_project.restype = C.c_int
    S.mxs_div_project.argtypes = [vp, vp, vp, C.c_double, vp, vp]
    S.mxs_magwave_apply_ex.restype = C.c_int
    S.mxs_magwave_apply_ex.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int,
                                       vp, vp, vp]
    _SOLVER = S
    return S


def _ck(rc):
    if rc != 0:
        raise MxError(load_library().mxg_last_error().decode())


def _scalar(a):
    a = complex(a)
    return (C.c_double * 2)(a.real, a.imag)


def _ints(v):
    v = [int(x) for x in v]
    return (C.c_int * len(v))(*v), len(v)


class Context:
    """One GPU + its streams (+ NCCL communicator): the MxComm of the B200 path (MxComm.hpp:14-37)."""

    def __init__(self, device=0):
        self._L = load_library()
        h = C.c_void_p()
        _ck(self._L.mxg_ctx_create(int(device), C.byref(h)))
        self.h = h

    @staticmethod
    def unique_id():
        buf = (C.c_ubyte * 128)()
        _ck(load_library().mxg_comm_unique_id(buf))
        return bytes(buf)

    def comm_init(self, rank, nranks, unique_id=None):
        buf = (C.c_ubyte * 128)(*unique_id) if unique_id is not None else None
        _ck(self._L.mxg_ctx_comm_init(self.h, rank, nranks, buf))

    def myPID(self):
        return self._L.mxg_ctx_rank(self.h)

    def numProc(self):
        return self._L.mxg_ctx_num_ranks(self.h)

    def sync(self):
        _ck(self._L.mxg_ctx_sync(self.h))

    def stream(self):
        return self._L.mxg_ctx_stream(self.h)

    def launch_count(self):
        return self._L.mxg_ctx_launch_count(self.h)

    def event_record(self, slot):
        _ck(self._L.mxg_ctx_event_record(self.h, slot))

    def event_elapsed_ms(self, a, b):
        ms = C.c_double()
        _ck(self._L.mxg_ctx_event_elapsed_ms(self.h, a, b, C.byref(ms)))
        return ms.value

    def close(self):
        if self.h:
            self._L.mxg_ctx_destroy(self.h)
            self.h = None


class MxMap:
    """MxMap(globalIndices, comm) (MxMap.hpp:22-103): this rank's owned GIDs, ascending."""

    def __init__(self, ctx, num_global, my_gids, components=1):
        """components > 1: multivectors on this map are stored component-major on the device (mxg_map_create_ordered;
        GID = comp + components * cell). from_host / to_host translate, so callers keep the reference order."""
        self.ctx = ctx
        self._L = ctx._L
        g = np.ascontiguousarray(my_gids, dtype=np.int64)
        h = C.c_void_p()
        self.perm = None
        if int(components) > 1:
            _ck(self._L.mxg_map_create_ordered(ctx.h, int(num_global), g.ctypes.data, len(g), int(components), C.byref(h)))
            perm = np.empty(len(g), dtype=np.int32)
            rc = self._L.mxg_map_get_order(h, perm.ctypes.data)
            _ck(min(rc, 0))
            if rc == 1:
                self.perm = perm.astype(np.int64)          # perm[device position] = reference local index
        else:
            _ck(self._L.mxg_map_create(ctx.h, int(num_global), g.ctypes.data, len(g), C.byref(h)))
        self.h = h
        self.gids = g

    def getNodeNumIndices(self):
        return self._L.mxg_map_local_size(self.h)

    def getGlobalNumIndices(self):
        return self._L.mxg_map_global_size(self.h)

    def __del__(self):
        try:
            if self.h:
                self._L.mxg_map_destroy(self.h)
        except Exception:
            pass


class MxMultiVector:
    """MxMultiVector / MxAnasaziMV (MxMultiVector.hpp:16-89, MxAnasaziMV.hpp:23-136)."""

    def __init__(self, map_, num_vecs, is_complex=False, _handle=None):
        self.map = map_
        self._L = map_._L
        if _handle is None:
            h = C.c_void_p()
            _ck(self._L.mxg_mv_create(map_.h, int(num_vecs), int(bool(is_complex)), C.byref(h)))
            _handle = h
        self.h = _handle
        self.is_complex = bool(self._L.mxg_mv_is_complex(self.h))
        self.dtype = np.complex128 if self.is_complex else np.float64

    # -- Anasazi::MultiVec surface -------------------------------------------------------
    def Clone(self, num_vecs):
        return MxMultiVector(self.map, num_vecs, self.is_complex)

    def CloneCopy(self, index=None):
        h = C.c_void_p()
        if index is None:
            _ck(self._L.mxg_mv_clone_copy(self.h, None, 0, C.byref(h)))
        else:
            arr, n = _ints(index)
            _ck(self._L.mxg_mv_clone_copy(self.h, arr, n, C.byref(h)))
        return MxMultiVector(self.map, 0, _handle=h)

    def CloneView(self, index):
        arr, n = _ints(index)
        h = C.c_void_p()
        _ck(self._L.mxg_mv_view(self.h, arr, n, C.byref(h)))
        return MxMultiVector(self.map, 0, _handle=h)

    CloneViewNonConst = CloneView

    def GetVecLength(self):
        return self._L.mxg_mv_global_length(self.h)

    def GetNumberVecs(self):
        return self._L.mxg_mv_num_cols(self.h)

    getNumVecs = GetNumberVecs

    def getLocalLength(self):
        return self._L.mxg_mv_local_length(self.h)

    def MvTimesMatAddMv(self, alpha, A, B, beta, ldb=None):
        """this = alpha*A*B + beta*this; B: host (k x b) array, or with ldb an (ldb x b) array of which the first k rows
        are read."""
        k = A.GetNumberVecs()
        Bh = np.asfortranarray(np.asarray(B, dtype=self.dtype).reshape(k if ldb is None else int(ldb), -1))
        _ck(self._L.mxg_mv_times_mat_add_mv(_scalar(alpha), A.h, Bh.ctypes.data, Bh.shape[0], _scalar(beta), self.h))

    def MvAddMv(self, alpha, A, beta, B):
        _ck(self._L.mxg_mv_add_mv(self.h, _scalar(alpha), A.h, _scalar(beta), B.h))

    def MvTransMv(self, alpha, A, ldb=None, out=None):
        """returns alpha * A^H * this as a host (k x b) array. With ldb, the product fills the first k rows of an (ldb x b)
        column-major array (`out`, whose other rows are left as they are, or a new zero array), which is returned."""
        k, b = A.GetNumberVecs(), self.GetNumberVecs()
        ldb = k if ldb is None else int(ldb)
        if out is None:
            out = np.zeros((ldb, b), dtype=self.dtype, order="F")
        if out.shape != (ldb, b) or out.dtype != self.dtype or not out.flags.f_contiguous:
            raise MxError("MvTransMv: out must be a column-major %d x %d %s array" % (ldb, b, np.dtype(self.dtype).name))
        _ck(self._L.mxg_mv_trans_mv(_scalar(alpha), A.h, self.h, out.ctypes.data, ldb))
        return out

    def trans_mv(self, alpha, X):
        """alpha * this^H * X."""
        return X.MvTransMv(alpha, self)

    def MvDot(self, A):
        out = np.zeros(self.GetNumberVecs(), dtype=self.dtype)
        _ck(self._L.mxg_mv_dot(A.h, self.h, out.ctypes.data))
        return out

    def dot(self, mv):
        """mv^dagger . this (MxMultiVector.hpp:58-61)."""
        return self.MvDot(mv)

    def MvNorm(self):
        out = np.zeros(self.GetNumberVecs(), dtype=np.float64)
        _ck(self._L.mxg_mv_norm2(self.h, out.ctypes.data))
        return out

    norm2 = MvNorm

    def SetBlock(self, A, index):
        arr, n = _ints(index)
        _ck(self._L.mxg_mv_set_block(self.h, A.h, arr, n))

    def MvScale(self, alpha):
        if np.ndim(alpha) == 0:
            _ck(self._L.mxg_mv_scale(self.h, _scalar(alpha)))
        else:
            a = np.ascontiguousarray(alpha, dtype=self.dtype)
            assert len(a) == self.GetNumberVecs()
            _ck(self._L.mxg_mv_scale_cols(self.h, a.ctypes.data))

    scale = MvScale

    def MvRandom(self, seed=12345):
        _ck(self._L.mxg_mv_random(self.h, int(seed)))

    random = MvRandom

    def MvInit(self, alpha):
        _ck(self._L.mxg_mv_fill(self.h, _scalar(alpha)))

    set = MvInit

    def conj(self):
        _ck(self._L.mxg_mv_conj(self.h))

    def update(self, a, A, s):
        _ck(self._L.mxg_mv_update(self.h, _scalar(a), A.h, _scalar(s)))

    def assign(self, src):
        _ck(self._L.mxg_mv_assign(self.h, src.h))

    def axpby_cols(self, alphas, A, betas, B):
        """this_j = alphas[j] * A_j + betas[j] * B_j (per-column scalars; A and / or B may be this)."""
        a = np.ascontiguousarray(alphas, dtype=self.dtype)
        b = np.ascontiguousarray(betas, dtype=self.dtype)
        assert len(a) == len(b) == self.GetNumberVecs()
        _ck(self._L.mxg_mv_axpby_cols(self.h, a.ctypes.data, A.h, b.ctypes.data, B.h))

    def remove_const_field(self):
        """removeConstField (MxGeoMultigridPrec.cpp:400-411): subtract each column's mean."""
        _ck(self._L.mxg_mv_remove_const_field(self.h))

    def zero_unused(self, fracs):
        """MxGridField::zeroUnusedComponents (MxGridField.cpp:548-576): zero the entries whose shape fraction is 0."""
        _ck(self._L.mxg_mv_zero_unused(self.h, fracs.h))

    def normalize(self):
        _ck(self._L.mxg_mv_normalize(self.h))

    # -- host transfers -------------------------------------------------------------------
    def from_host(self, arr):
        n, b = self.getLocalLength(), self.GetNumberVecs()
        a = np.asfortranarray(np.asarray(arr, dtype=self.dtype).reshape(n, b))
        perm = getattr(self.map, "perm", None)
        if perm is not None:                               # ordered map: the device stores row perm[i] at position i
            a = np.asfortranarray(a[perm, :])
        _ck(self._L.mxg_mv_upload(self.h, a.ctypes.data, n))

    def to_host(self, out=None):
        n, b = self.getLocalLength(), self.GetNumberVecs()
        perm = getattr(self.map, "perm", None)
        if perm is not None:
            dev = np.empty((n, b), dtype=self.dtype, order="F")
            _ck(self._L.mxg_mv_download(self.h, dev.ctypes.data, n))
            if out is None:
                out = np.empty((n, b), dtype=self.dtype, order="F")
            out[perm, :] = dev
            return out
        if out is None:
            out = np.empty((n, b), dtype=self.dtype, order="F")
        _ck(self._L.mxg_mv_download(self.h, out.ctypes.data, n))
        return out

    def to_grid(self, col, gid_lo, gid_hi):
        """Column `col` in the dense [cell][comp] layout MxIO::save writes (src/MxIO.cpp:166-221), zeros at masked DOFs."""
        n = int(gid_hi) - int(gid_lo)
        re = np.empty(n, dtype=np.float64)
        im = np.empty(n, dtype=np.float64) if self.is_complex else None
        _ck(self._L.mxg_mv_to_grid(self.h, int(col), int(gid_lo), int(gid_hi), re.ctypes.data,
                                   im.ctypes.data if im is not None else None))
        return re + 1j * im if im is not None else re

    def col_ptr(self, j):
        return self._L.mxg_mv_col_ptr(self.h, j)

    def __del__(self):
        try:
            if self.h:
                self._L.mxg_mv_destroy(self.h)
        except Exception:
            pass


MxAnasaziMV = MxMultiVector


class MxCrsMatrix:
    """MxCrsMatrix (MxCrsMatrix.hpp:14-82): host assembly by insertRowValues, device apply."""

    def __init__(self, row_map, col_map=None, is_complex=False):
        self.row_map = row_map
        self.col_map = col_map if col_map is not None else row_map
        self.is_complex = bool(is_complex)
        self._L = row_map._L
        self._rows = {}
        self.h = None

    def insertRowValues(self, row, cols, vals):
        """Global indices, as in the reference (MxCrsMatrix.hpp:31-36); duplicates are summed."""
        self._rows.setdefault(int(row), []).extend(zip([int(c) for c in cols], list(vals)))

    def fillComplete(self, domain_map=None, range_map=None, layout=None):
        if domain_map is not None:
            self.col_map = domain_map
        gids = self.row_map.gids
        rowptr = np.zeros(len(gids) + 1, dtype=np.int64)
        cols, vals = [], []
        for i, g in enumerate(gids):
            ent = self._rows.get(int(g), [])
            cols.extend(c for c, _ in ent)
            vals.extend(v for _, v in ent)
            rowptr[i + 1] = len(cols)
        self._finish(rowptr, np.asarray(cols, dtype=np.int64),
                     np.asarray(vals, dtype=np.complex128 if self.is_complex else np.float64), layout)
        self._rows = {}

    @classmethod
    def from_csr(cls, row_map, domain_map, rowptr, col_gids, vals, layout=None):
        A = cls(row_map, domain_map, np.iscomplexobj(vals))
        A._finish(np.ascontiguousarray(rowptr, dtype=np.int64), np.ascontiguousarray(col_gids, dtype=np.int64),
                  np.ascontiguousarray(vals, dtype=np.complex128 if A.is_complex else np.float64), layout)
        return A

    def _finish(self, rowptr, cols, vals, layout):
        h = C.c_void_p()
        if layout is None:
            _ck(self._L.mxg_crs_create(self.row_map.h, self.col_map.h, rowptr.ctypes.data, cols.ctypes.data,
                                       vals.ctypes.data, int(self.is_complex), C.byref(h)))
        else:
            _ck(self._L.mxg_crs_create_opts(self.row_map.h, self.col_map.h, rowptr.ctypes.data, cols.ctypes.data,
                                            vals.ctypes.data, int(self.is_complex), int(layout), C.byref(h)))
        self.h = h

    def isFilled(self):
        return self.h is not None

    def getDomainMap(self):
        return self.col_map

    def getRangeMap(self):
        return self.row_map

    def apply(self, x, y):
        _ck(self._L.mxg_crs_apply(self.h, x.h, y.h))

    def apply_host_batch(self, xs, ys):
        """ys[i] = A xs[i] for host arrays (one column each; pinned arrays make the copies asynchronous); uploads,
        applies and downloads are pipelined inside the library."""
        n = len(xs)
        assert len(ys) == n
        xp = (C.c_void_p * n)(*[a.ctypes.data for a in xs])
        yp = (C.c_void_p * n)(*[a.ctypes.data for a in ys])
        _ck(self._L.mxg_crs_apply_host_batch(self.h, n, xp, yp))

    def apply_axpby(self, alpha, x, beta, y):
        _ck(self._L.mxg_crs_apply_axpby(self.h, _scalar(alpha), x.h, _scalar(beta), y.h))

    def apply_timed(self, x, y):
        ms = (C.c_double * 4)()
        _ck(self._L.mxg_crs_apply_timed(self.h, x.h, y.h, ms))
        return {"dict_ms": ms[0], "sell_ms": ms[1], "pre_ms": ms[2], "total_ms": ms[3]}

    def trace_apply(self, x, y):
        """One multi-rank apply with %globaltimer marks: ns since the first mark for pack / interior / boundary roles."""
        out = (C.c_double * 10)()
        _ck(self._L.mxg_crs_trace(self.h, 1, out))
        self.apply(x, y)
        _ck(self._L.mxg_crs_trace(self.h, 0, out))
        names = ["pack", "interior_dict", "interior_sell", "boundary_wait", "boundary_rows"]
        return {n: (out[2 * i], out[2 * i + 1]) for i, n in enumerate(names)}

    def stats(self):
        out = (C.c_int64 * 8)()
        _ck(self._L.mxg_crs_stats(self.h, out))
        keys = ["rows", "nnz", "dict_rows", "patterns", "device_bytes", "ghosts", "ghost_rows", "ell_entries"]
        return dict(zip(keys, list(out)))

    def __del__(self):
        try:
            if self.h:
                self._L.mxg_crs_destroy(self.h)
        except Exception:
            pass


def pinned_array(shape, dtype=np.float64):
    """numpy array backed by cudaMallocHost memory (freed when the array is collected)."""
    L = load_library()
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = L.mxg_host_alloc(n)
    if not p:
        raise MxError(L.mxg_last_error().decode())
    buf = (C.c_ubyte * n).from_address(p)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape, order="F")
    _PINNED[id(buf)] = (buf, p)
    return arr


_PINNED = {}


def hash_uniform(seed, gids, col, part=0):
    """Host mirror of the counter-based generator behind MvRandom (mxg_mvops.cu: hashUniform)."""
    with np.errstate(over="ignore"):
        g = np.asarray(gids, dtype=np.uint64)
        z = (np.uint64(seed) ^ (g * np.uint64(0x9E3779B97F4A7C15))
             ^ np.uint64(((col + 1) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF)
             ^ np.uint64((part * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF))
        z ^= z >> np.uint64(30)
        z *= np.uint64(0xBF58476D1CE4E5B9)
        z ^= z >> np.uint64(27)
        z *= np.uint64(0x94D049BB133111EB)
        z ^= z >> np.uint64(31)
        return 2.0 * ((z >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)) - 1.0


def diag_mult(y, d, x):
    """y = d .* x with d a one-column multivector (mRhs = dmA; MxMagWaveOp.cpp:865,895)."""
    _ck(load_library().mxg_mv_diag_mult(y.h, d.h, x.h))


class MxGeoMultigridPrec:
    """GPU V-cycle / FMG preconditioner (spec: reference src/MxGeoMultigridPrec.cpp; dead code there).

    ops[l]: level operators fine -> coarse; restrictors[l]: level l -> l+1; prolongators[l]: l+1 -> l.
    Keyword parameters mirror the reference's "linear solver : ..." keys (MxGeoMultigridPrec.cpp:100-108).
    """

    def __init__(self, ctx, ops, restrictors, prolongators, smoother_sweeps=2, cycles=1, eig_ratio=30.0,
                 coarse_degree=30, coarse_eig_ratio=1000.0, full_multigrid=False, power_iterations=30, remove_const_field=False):
        self._L = load_library()
        self._keep = (list(ops), list(restrictors), list(prolongators))
        p = GmgParams()
        self._L.mxg_gmg_default_params(C.byref(p))
        p.smoother_degree, p.cycles, p.eig_ratio = int(smoother_sweeps), int(cycles), float(eig_ratio)
        p.coarse_degree, p.coarse_eig_ratio = int(coarse_degree), float(coarse_eig_ratio)
        p.full_multigrid, p.power_iterations = int(bool(full_multigrid)), int(power_iterations)
        p.remove_const_field = int(bool(remove_const_field))
        n = len(ops)
        arr = lambda xs: (C.c_void_p * max(len(xs), 1))(*[x.h for x in xs])
        h = C.c_void_p()
        _ck(self._L.mxg_gmg_create(ctx.h, n, arr(ops), arr(restrictors), arr(prolongators), C.byref(p), C.byref(h)))
        self.h = h
        self.nlevels = n

    def ApplyInverse(self, b, x):
        _ck(self._L.mxg_gmg_apply(self.h, b.h, x.h))

    def info(self, level):
        out = (C.c_double * 4)()
        _ck(self._L.mxg_gmg_info(self.h, level, out))
        return {"rows": int(out[0]), "nnz": int(out[1]), "lambda_max": out[2], "spmm_count": int(out[3])}

    def __del__(self):
        try:
            if self.h:
                self._L.mxg_gmg_destroy(self.h)
        except Exception:
            pass


class MxSolver:
    """Block eigensolver driver (reference: src/MxSolver.cpp:22-239 driving Anasazi): lowest eigenpairs of
    A x = theta M x with an optional multigrid preconditioner. The loop runs in C++ (include/mx/MxSolver.hpp).
    Real symmetric pencils, or Hermitian ones (complex operator of a Bloch-periodic simulation: complex multivectors,
    m_diag a complex one-column multivector)."""

    def __init__(self, ctx, A, m_diag=None, prec=None, nev=10, block_size=0, tol=1e-8, max_iters=300, verbose=0, seed=12345,
                 projection=None):
        """projection: dict(divB=, gradPsi=, scaLapl=, sca_prec=None, tol_w=..., tol_x=..., tol_init=..., reproject_ratio=...)
        constrains the iteration to the divergence-free fields (MxMagWaveOp.cpp:893-924): only Maxwell modes are returned."""
        self._S = load_solver()
        self.ctx, self.A, self.m_diag, self.prec = ctx, A, m_diag, prec
        self.projection = projection
        p = SolverParams()
        self._S.mxs_default_params(C.byref(p))
        p.nev, p.block_size, p.tol, p.max_iters, p.verbose, p.seed = int(nev), int(block_size), float(tol), int(max_iters), int(verbose), int(seed)
        if p.block_size <= 0:
            p.block_size = nev + max(4, nev // 2)
        self.params = p

    def solve(self, X=None):
        m = self.params.block_size
        if X is None:
            X = MxMultiVector(self.A.row_map, m, getattr(self.A, "is_complex", False))
            self.params.random_init = 1
        else:
            self.params.random_init = 0
        ev = np.zeros(m)
        rs = np.zeros(m)
        info = (C.c_int64 * 4)()
        sec = C.c_double()
        if self.projection is None:
            rc = self._S.mxs_lobpcg(self.ctx.h, self.A.h, self.m_diag.h if self.m_diag is not None else None,
                                    self.prec.h if self.prec is not None else None, X.h, C.byref(self.params),
                                    ev.ctypes.data, rs.ctypes.data, info, C.byref(sec))
            self.violation = None
        else:
            pr = self.projection
            P = Projection()
            P.divB, P.gradPsi, P.scaLapl = pr["divB"].h, pr["gradPsi"].h, pr["scaLapl"].h
            P.sca_prec = pr["sca_prec"].h if pr.get("sca_prec") is not None else None
            P.tol_init, P.tol_w, P.tol_x = float(pr.get("tol_init", 0)), float(pr.get("tol_w", 0)), float(pr.get("tol_x", 0))
            P.reproject_ratio, P.max_iters = float(pr.get("reproject_ratio", 0)), int(pr.get("max_iters", 0))
            P.max_iters_w = int(pr.get("max_iters_w", 0))
            info = (C.c_int64 * 8)()
            viol = np.zeros(m)
            rc = self._S.mxs_lobpcg_projected(self.ctx.h, self.A.h, self.m_diag.h if self.m_diag is not None else None,
                                              self.prec.h if self.prec is not None else None, C.byref(P), X.h, C.byref(self.params),
                                              ev.ctypes.data, rs.ctypes.data, viol.ctypes.data, info, C.byref(sec))
            self.violation = viol
            self.projected_columns, self.reprojections, self.proj_cg_iters, self.proj_calls = info[4], info[5], info[6], info[7]
        if rc != 0:
            raise MxError(self._S.mxs_last_error().decode())
        self.eigenvalues, self.residuals, self.eigenvectors = ev, rs, X
        self.iterations, self.converged, self.apply_a, self.apply_prec = info[0], info[1], info[2], info[3]
        self.seconds = sec.value
        return ev[: self.params.nev]

    def check(self, div_op=None, A=None):
        """checkEigensolution / checkDivergences (MxMagWaveOp.cpp:1118-1234). A: operator of the residual check (the
        reference uses curlCurl there, not the vector Laplacian it solves with); default = the solver's own operator."""
        m = self.params.block_size
        res, div = np.zeros(m), np.zeros(m)
        rc = self._S.mxs_check_eigensolution(self.ctx.h, (A if A is not None else self.A).h, self.m_diag.h if self.m_diag is not None else None,
                                             div_op.h if div_op is not None else None, self.eigenvectors.h,
                                             self.eigenvalues.ctypes.data, res.ctypes.data, div.ctypes.data)
        if rc != 0:
            raise MxError(self._S.mxs_last_error().decode())
        return res, div


class MxMagWaveOp:
    """The shift-invert operator the reference hands to Anasazi (src/MxMagWaveOp.cpp:825-943):
    y = P (L - sigma M)^-1 M x, with the divergence-cleaning projection P. Inner solves: block PCG on the GPU."""

    LIN_SOLVERS = {"cg": 0, "bicgstab": 1, "gmres": 2}   # "linear solver : type" (MxMagWaveOp.cpp:326-338)

    def __init__(self, ctx, vec_lapl, m_diag, div_b=None, grad_psi=None, sca_lapl=None, vec_prec=None, sca_prec=None,
                 shift=0.0, lin_tol=1e-10, lin_solver="cg", lin_basis=20, max_lin_iters=1000):
        self._S = load_solver()
        self.ctx, self.L, self.m, self.D, self.G, self.S = ctx, vec_lapl, m_diag, div_b, grad_psi, sca_lapl
        self.vec_prec, self.sca_prec, self.shift, self.lin_tol = vec_prec, sca_prec, float(shift), float(lin_tol)
        self.has_curl_null = div_b is not None
        self.lin_solver, self.lin_basis, self.max_lin_iters = self.LIN_SOLVERS[lin_solver], int(lin_basis), int(max_lin_iters)
        self.num_vec_lin_iters = self.num_sca_lin_iters = self.num_applies = 0

    def Apply(self, x, y):
        h = lambda o: o.h if o is not None else None
        info = (C.c_int64 * 2)()
        rc = self._S.mxs_magwave_apply_ex(self.ctx.h, self.L.h, self.m.h, h(self.D), h(self.G), h(self.S), h(self.vec_prec),
                                          h(self.sca_prec), self.shift, self.lin_tol, int(self.has_curl_null), self.lin_solver,
                                          self.lin_basis, self.max_lin_iters, x.h, y.h, info)
        if rc != 0:
            raise MxError(self._S.mxs_last_error().decode())
        self.num_applies += 1
        self.num_vec_lin_iters += info[0]
        self.num_sca_lin_iters += info[1]


def div_project(ctx, m_diag, X, divB, gradPsi, scaLapl, sca_prec=None, tol=1e-10, max_iters=500):
    """X <- P X = X + gradPsi scaLapl^-1 divB M X (MxMagWaveOp.cpp:893-924); returns the inner CG iteration count."""
    S = load_solver()
    P = Projection()
    P.divB, P.gradPsi, P.scaLapl = divB.h, gradPsi.h, scaLapl.h
    P.sca_prec = sca_prec.h if sca_prec is not None else None
    P.max_iters = int(max_iters)
    info = (C.c_int64 * 1)()
    if S.mxs_div_project(ctx.h, m_diag.h if m_diag is not None else None, C.byref(P), float(tol), X.h, info) != 0:
        raise MxError(S.mxs_last_error().decode())
    return int(info[0])


def mag_to_elec(ctx, curl_b, inv_eps, mag, elec):
    """MxMagWaveOp::magToElec (src/MxMagWaveOp.cpp:1237-1250): elec = [invEps] curlB mag."""
    S = load_solver()
    if S.mxs_mag_to_elec(ctx.h, curl_b.h, inv_eps.h if inv_eps is not None else None, mag.h, elec.h) != 0:
        raise MxError(S.mxs_last_error().decode())


def eigvals_to_freqs(eigvals, shift=0.0, invert=False):
    """MxMagWaveOp::eigValsToFreqs (src/MxMagWaveOp.cpp:1252-1271): complex frequencies in Hz."""
    S = load_solver()
    ev = np.ascontiguousarray(np.asarray(eigvals, dtype=np.complex128))
    re, im = np.ascontiguousarray(ev.real), np.ascontiguousarray(ev.imag)
    fre, fim = np.empty_like(re), np.empty_like(re)
    if S.mxs_eigvals_to_freqs(re.ctypes.data, im.ctypes.data, len(re), float(shift), int(invert), fre.ctypes.data,
                              fim.ctypes.data) != 0:
        raise MxError(S.mxs_last_error().decode())
    return fre + 1j * fim
