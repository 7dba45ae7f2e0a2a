"""ctypes veneer of the operator-assembly entry points (include/mxasm.h): shapes, the simulation set-up (fields, DOF
maps, cut-cell fractions) and the device CRS algebra that chains the Yee operators.

`AssemblyAPI(lib, prefix)` binds one library: the product binds libmxgpu.so with the `mxg_` prefix (see `gpu_api()`);
the CPU suite binds the replay build of the same sources (tests/cpp/asm_replay.cpp, prefix `mxr_`) to pin the logic
against the oracle without a GPU. Nothing here computes: every call lands in the library.
"""
import ctypes as C

import numpy as np

PERIODIC, ZERO, CONSTANT, PEC, PMC = 0, 1, 2, 3, 4
FIELDS = ("bfield", "efield", "psifield")


class AssemblyError(RuntimeError):
    pass


def _d3(v):
    return (C.c_double * 3)(*[float(x) for x in v])


def _i3(v):
    return (C.c_int * 3)(*[int(x) for x in v])


class AssemblyAPI:
    def __init__(self, lib, prefix, last_error):
        self.lib, self.prefix, self._last_error = lib, prefix, last_error
        vp, i64, i32, dbl = C.c_void_p, C.c_int64, C.c_int, C.c_double
        pvp, d3, i3 = C.POINTER(C.c_void_p), C.POINTER(C.c_double), C.POINTER(C.c_int)
        sig = {
            "sim_create": [vp, i3, d3, d3, i3, i3, d3, dbl, i32, pvp],
            "sim_destroy": [vp],
            "sim_set_pec_fractions": [vp, C.c_char_p, vp],
            "sim_set_pec_shape": [vp, vp],
            "sim_add_dielectric": [vp, vp, vp],
            "sim_setup": [vp],
            "sim_map_size": [vp, C.c_char_p, C.POINTER(i64), C.POINTER(i64)],
            "sim_map_copy": [vp, C.c_char_p, vp],
            "sim_fractions": [vp, C.c_char_p, vp],
            "sim_op": [vp, C.c_char_p, i32, vp, vp, pvp],
            "sim_op_rows": [vp, C.c_char_p, i32, vp, vp, i64, i64, pvp],
            "dcsr_upload": [vp, C.c_char_p, C.c_char_p, i64, i64, vp, vp, vp, i32, pvp],
            "dcsr_multiply": [vp, vp, pvp],
            "dcsr_add": [vp, d3, vp, d3, i32, pvp],
            "dcsr_purge": [vp, pvp],
            "dcsr_scale": [vp, d3],
            "dcsr_transpose": [vp, pvp],
            "sim_interpolator": [vp, vp, C.c_char_p, i32, pvp],
            "sim_interpolator_rows": [vp, vp, C.c_char_p, i32, i64, i64, pvp],
            "sim_interpolator_transpose_rows": [vp, vp, C.c_char_p, i32, i64, i64, pvp],
            "dcsr_shape": [vp, C.POINTER(i64)],
            "dcsr_rows": [vp, C.POINTER(i64)],
            "dcsr_download": [vp, i64, i64, vp, vp, vp],
            "dcsr_destroy": [vp],
            "shape_cylinder": [dbl, d3, d3, pvp],
            "shape_sphere": [dbl, d3, pvp],
            "shape_halfspace": [d3, d3, pvp],
            "shape_slab": [dbl, d3, d3, pvp],
            "shape_ellipsoid": [d3, d3, pvp],
            "shape_torus": [dbl, dbl, d3, d3, pvp],
            "shape_cone": [dbl, d3, d3, pvp],
            "shape_intersection": [pvp, i32, pvp],
            "shape_union": [pvp, i32, pvp],
            "shape_subtract": [vp, pvp, i32, pvp],
            "shape_mirror": [vp, d3, d3, pvp],
            "shape_repeat": [vp, d3, d3, dbl, i32, i32, pvp],
            "shape_translate": [vp, d3],
            "shape_rotate": [vp, d3, dbl, vp],
            "shape_scale": [vp, d3, d3],
            "shape_reflect": [vp, d3, d3],
            "shape_invert": [vp],
            "shape_eval": [vp, d3, d3, d3],
            "shape_destroy": [vp],
        }
        self.fn = {}
        for name, args in sig.items():
            f = getattr(lib, prefix + name)
            f.restype = C.c_int
            f.argtypes = args
            self.fn[name] = f

    def call(self, name, *args):
        rc = self.fn[name](*args)
        if rc != 0:
            msg = self._last_error()
            raise AssemblyError("%s%s failed (%d): %s" % (self.prefix, name, rc, msg.decode() if isinstance(msg, bytes) else msg))

    # ---- shapes (MxShape and its subclasses) ----
    def _new_shape(self, name, *args, keep=()):
        h = C.c_void_p()
        self.call(name, *args, C.byref(h))
        return Shape(self, h, keep)

    def cylinder(self, r, axis, loc):
        return self._new_shape("shape_cylinder", float(r), _d3(axis), _d3(loc))

    def sphere(self, r, loc):
        return self._new_shape("shape_sphere", float(r), _d3(loc))

    def halfspace(self, point, normal):
        return self._new_shape("shape_halfspace", _d3(point), _d3(normal))

    def slab(self, thickness, normal, loc):
        return self._new_shape("shape_slab", float(thickness), _d3(normal), _d3(loc))

    def ellipsoid(self, loc, axes):
        return self._new_shape("shape_ellipsoid", _d3(loc), _d3(axes))

    def torus(self, major_radius, minor_radius, axis, loc):
        return self._new_shape("shape_torus", float(major_radius), float(minor_radius), _d3(axis), _d3(loc))

    def cone(self, angle, axis, vertex):
        return self._new_shape("shape_cone", float(angle), _d3(axis), _d3(vertex))

    def _list(self, shapes):
        return (C.c_void_p * len(shapes))(*[s.handle for s in shapes])

    def intersection(self, shapes):
        return self._new_shape("shape_intersection", self._list(shapes), len(shapes))

    def union(self, shapes):
        return self._new_shape("shape_union", self._list(shapes), len(shapes))

    def subtract(self, base, removed):
        removed = [removed] if isinstance(removed, Shape) else list(removed)
        return self._new_shape("shape_subtract", base.handle, self._list(removed), len(removed))

    def mirror(self, shape, normal, point):
        return self._new_shape("shape_mirror", shape.handle, _d3(normal), _d3(point))

    def repeat(self, shape, origin, direction, step, num_pos, num_neg):
        return self._new_shape("shape_repeat", shape.handle, _d3(origin), _d3(direction), float(step), int(num_pos), int(num_neg))

    # ---- simulation ----
    def sim(self, ctx_handle, n, origin=(0.0, 0.0, 0.0), size=(1.0, 1.0, 1.0), lower=None, upper=None, phase_shifts=None,
            dm_frac=0.0, literal_upper_periodic_e=False):
        n = (n,) * 3 if np.isscalar(n) else tuple(n)
        h = C.c_void_p()
        self.call("sim_create", ctx_handle, _i3(n), _d3(origin), _d3(size), _i3(lower or (PERIODIC,) * 3),
                  _i3(upper or (PERIODIC,) * 3), _d3(phase_shifts or (0.0, 0.0, 0.0)), float(dm_frac),
                  1 if literal_upper_periodic_e else 0, C.byref(h))
        return Sim(self, h, n, phase_shifts is not None and any(p != 0 for p in phase_shifts))


class Shape:
    """Host-side CSG shape (copied into composites, so parts may be released or transformed afterwards)."""

    def __init__(self, api, handle, keep=()):
        self.api, self.handle = api, handle

    def translate(self, v):
        self.api.call("shape_translate", self.handle, _d3(v))
        return self

    def rotate(self, axis, angle, pivot=None):
        p = _d3(pivot) if pivot is not None else None
        self.api.call("shape_rotate", self.handle, _d3(axis), float(angle), C.cast(p, C.c_void_p) if p is not None else None)
        return self

    def scale(self, magnitudes, origin=(0.0, 0.0, 0.0)):
        self.api.call("shape_scale", self.handle, _d3(magnitudes), _d3(origin))
        return self

    def reflect(self, normal, point):
        self.api.call("shape_reflect", self.handle, _d3(normal), _d3(point))
        return self

    def invert(self):
        self.api.call("shape_invert", self.handle)
        return self

    def func(self, p):
        f = (C.c_double * 3)()
        self.api.call("shape_eval", self.handle, _d3(p), f, None)
        return f[0]

    def grad(self, p):
        g = (C.c_double * 3)()
        self.api.call("shape_eval", self.handle, _d3(p), None, g)
        return np.array(g[:])

    def __del__(self):
        try:
            if self.handle:
                self.api.fn["shape_destroy"](self.handle)
                self.handle = None
        except Exception:
            pass


class Sim:
    """MxEMSim (MxEMSim.cpp:54-199): grid, boundary conditions, optional PEC shape, DOF maps; operators by name."""

    def __init__(self, api, handle, n, is_complex):
        self.api, self.handle, self.n, self.is_complex = api, handle, n, is_complex
        self._setup = False

    def set_pec_shape(self, shape):
        self.api.call("sim_set_pec_shape", self.handle, shape.handle)
        self._setup = False
        return self

    def add_dielectric(self, shape, eps):
        """MxEMSim::addDielectric: a shape filled with the permittivity tensor eps (scalar, 3 diagonal values or 3x3, real or complex)."""
        e = np.asarray(eps, dtype=np.complex128)
        if e.ndim == 0:
            e = np.eye(3) * e
        elif e.ndim == 1:
            e = np.diag(e)
        e = np.ascontiguousarray(e.reshape(3, 3).astype(np.complex128))
        self.api.call("sim_add_dielectric", self.handle, shape.handle, e.ctypes.data)
        self._setup = False
        return self

    def set_pec_fractions(self, field, fracs):
        a = np.ascontiguousarray(fracs, dtype=np.float64)
        ncomp = 1 if field == "psifield" else 3
        want = (self.n[0] + 3) * (self.n[1] + 3) * (self.n[2] + 3) * ncomp
        if a.size != want:
            raise ValueError("fractions of %s need %d values (guarded block x components), got %d" % (field, want, a.size))
        self.api.call("sim_set_pec_fractions", self.handle, field.encode(), a.ctypes.data)
        self._setup = False
        return self

    def setup(self):
        self.api.call("sim_setup", self.handle)
        self._setup = True
        return self

    def map_size(self, field):
        nl, ng = C.c_int64(), C.c_int64()
        self.api.call("sim_map_size", self.handle, field.encode(), C.byref(nl), C.byref(ng))
        return nl.value, ng.value

    def num_global(self, field):
        return self.map_size(field)[1]

    def map(self, field):
        out = np.empty(self.map_size(field)[0], dtype=np.int64)
        self.api.call("sim_map_copy", self.handle, field.encode(), out.ctypes.data)
        return out

    def fracs(self, field):
        ncomp = 1 if field == "psifield" else 3
        out = np.empty((self.n[0] + 3) * (self.n[1] + 3) * (self.n[2] + 3) * ncomp)
        self.api.call("sim_fractions", self.handle, field.encode(), out.ctypes.data)
        return out

    def op(self, name, is_complex=None, inv_eps=None, inv_eps_vol_ave=None, rows=None):
        """A named operator; rows=(begin, end) assembles only those rows of its row map (bit for bit the same rows)."""
        if not self._setup:
            self.setup()
        cplx = self.is_complex if is_complex is None else bool(is_complex)
        h = C.c_void_p()
        eps = (inv_eps.handle if inv_eps is not None else None, inv_eps_vol_ave.handle if inv_eps_vol_ave is not None else None)
        if rows is None:
            self.api.call("sim_op", self.handle, name.encode(), 1 if cplx else 0, *eps, C.byref(h))
        else:
            self.api.call("sim_op_rows", self.handle, name.encode(), 1 if cplx else 0, *eps, int(rows[0]), int(rows[1]), C.byref(h))
        return DeviceCsr(self, h)

    def _setup_both(self, coarse):
        if not self._setup:
            self.setup()
        if not coarse._setup:
            coarse.setup()

    def interpolator_from(self, coarse, field="bfield", is_complex=None, rows=None):
        """MxGridFieldInterpolator: `field` of the simulation `coarse` interpolated at this simulation's DOFs (rows=(begin, end):
        only those rows of this simulation's map)."""
        self._setup_both(coarse)
        cplx = self.is_complex if is_complex is None else bool(is_complex)
        h = C.c_void_p()
        if rows is None:
            self.api.call("sim_interpolator", coarse.handle, self.handle, field.encode(), 1 if cplx else 0, C.byref(h))
        else:
            self.api.call("sim_interpolator_rows", coarse.handle, self.handle, field.encode(), 1 if cplx else 0, int(rows[0]),
                          int(rows[1]), C.byref(h))
        m = DeviceCsr(self, h)
        m.col_sim = coarse
        return m

    def interpolator_transpose(self, coarse, field="bfield", is_complex=None, rows=None):
        """The rows (begin, end) of the coarse map of interpolator_from(coarse, field)'s conjugate transpose (the restriction
        before its 1/8 scaling), generating the interpolator on the fine rows that reach them only. rows=None: all rows."""
        self._setup_both(coarse)
        cplx = self.is_complex if is_complex is None else bool(is_complex)
        if rows is None:
            rows = (0, coarse.map_size(field)[0])
        h = C.c_void_p()
        self.api.call("sim_interpolator_transpose_rows", coarse.handle, self.handle, field.encode(), 1 if cplx else 0, int(rows[0]),
                      int(rows[1]), C.byref(h))
        m = DeviceCsr(self, h)
        m.row_sim, m.col_sim = coarse, self
        return m

    def upload(self, row_field, col_field, rowptr, col, val, ncols):
        """Host CSR with local column indices -> device (operators still generated on the host, e.g. the dielectric invEps)."""
        rowptr = np.ascontiguousarray(rowptr, dtype=np.int64)
        col = np.ascontiguousarray(col, dtype=np.int32)
        cplx = np.iscomplexobj(val)
        val = np.ascontiguousarray(val, dtype=np.complex128 if cplx else np.float64)
        h = C.c_void_p()
        self.api.call("dcsr_upload", self.handle, row_field.encode() if row_field else None, col_field.encode() if col_field else None,
                      len(rowptr) - 1, int(ncols), rowptr.ctypes.data, col.ctypes.data, val.ctypes.data, 1 if cplx else 0, C.byref(h))
        return DeviceCsr(self, h)

    def __del__(self):
        try:
            if self.handle:
                self.api.fn["sim_destroy"](self.handle)
                self.handle = None
        except Exception:
            pass


class DeviceCsr:
    """A CRS matrix resident on the device (local column indices, rows in the reference's entry order)."""

    def __init__(self, sim, handle):
        self.sim, self.api, self.handle = sim, sim.api, handle
        s = (C.c_int64 * 6)()
        self.api.call("dcsr_shape", handle, s)
        self.nrows, self.ncols, self.nnz, self.is_complex = s[0], s[1], s[2], bool(s[3])
        self.row_field = FIELDS[s[4]] if s[4] >= 0 else None
        self.col_field = FIELDS[s[5]] if s[5] >= 0 else None
        r = (C.c_int64 * 2)()
        self.api.call("dcsr_rows", handle, r)
        self.row_begin = r[0]          # map position of the first stored row (nrows counts the stored rows)

    def arrays(self, row_begin=0, row_end=None):
        """Stored rows [row_begin, row_end): rowptr rebased to 0, column positions in the whole column map, values."""
        row_end = self.nrows if row_end is None else row_end
        rowptr = np.empty(row_end - row_begin + 1, dtype=np.int64)
        self.api.call("dcsr_download", self.handle, row_begin, row_end, rowptr.ctypes.data, None, None)
        cnt = int(rowptr[-1])
        col = np.empty(cnt, dtype=np.int32)
        val = np.empty(cnt, dtype=np.complex128 if self.is_complex else np.float64)
        self.api.call("dcsr_download", self.handle, row_begin, row_end, rowptr.ctypes.data, col.ctypes.data, val.ctypes.data)
        return rowptr, col, val

    def __matmul__(self, other):
        h = C.c_void_p()
        self.api.call("dcsr_multiply", self.handle, other.handle, C.byref(h))
        return DeviceCsr(self.sim, h)

    def add(self, sa, other, sb, purge=False):
        h = C.c_void_p()
        sa, sb = complex(sa), complex(sb)
        self.api.call("dcsr_add", self.handle, _d3((sa.real, sa.imag, 0)), other.handle, _d3((sb.real, sb.imag, 0)),
                      1 if purge else 0, C.byref(h))
        return DeviceCsr(self.sim, h)

    def transpose(self, scale=None):
        h = C.c_void_p()
        self.api.call("dcsr_transpose", self.handle, C.byref(h))
        t = DeviceCsr(self.sim, h)
        t.col_sim = self.sim                      # keep both simulations alive
        t.row_sim = getattr(self, "col_sim", self.sim)
        if scale is not None:
            t.scale(scale)
        return t

    def purge(self):
        h = C.c_void_p()
        self.api.call("dcsr_purge", self.handle, C.byref(h))
        return DeviceCsr(self.sim, h)

    def scale(self, s):
        s = complex(s)
        self.api.call("dcsr_scale", self.handle, _d3((s.real, s.imag, 0)))
        return self

    def __del__(self):
        try:
            if self.handle:
                self.api.fn["dcsr_destroy"](self.handle)
                self.handle = None
        except Exception:
            pass


# ---- the product binding: libmxgpu.so ----------------------------------------------------------------------------
_GPU_API = None


def gpu_api():
    """The mxg_* entry points of libmxgpu.so (include/mxasm.h). Fails loudly when the library is missing."""
    global _GPU_API
    if _GPU_API is None:
        import maxwell_b200 as mx
        L = mx.load_library()
        api = AssemblyAPI(L, "mxg_", L.mxg_last_error)
        L.mxg_crs_create_from_dcsr.restype = C.c_int
        L.mxg_crs_create_from_dcsr.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        L.mxg_sim_make_map.restype = C.c_int
        L.mxg_sim_make_map.argtypes = [C.c_void_p, C.c_char_p, C.c_int64, C.c_int64, C.POINTER(C.c_void_p)]
        L.mxg_asm_memory.restype = C.c_int
        L.mxg_asm_memory.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.c_int]
        _GPU_API = api
    return _GPU_API


def gpu_sim(ctx, n, **kw):
    """A device-resident simulation on the context's GPU (arguments as AssemblyAPI.sim)."""
    sim = gpu_api().sim(ctx.h, n, **kw)
    sim.ctx = ctx
    return sim


def make_map(sim, field, begin=0, end=-1):
    """Rows [begin, end) of a field's DOF map as an MxMap of the simulation's context."""
    import maxwell_b200 as mx
    api = sim.api
    h = C.c_void_p()
    rc = api.lib.mxg_sim_make_map(sim.handle, field.encode(), int(begin), int(end), C.byref(h))
    if rc != 0:
        raise AssemblyError("mxg_sim_make_map failed (%d): %s" % (rc, api.lib.mxg_last_error().decode()))
    m = mx.MxMap.__new__(mx.MxMap)
    m.ctx, m._L, m.h = sim.ctx, sim.ctx._L, h
    gids = sim.map(field)
    m.gids = gids[begin:(len(gids) if end < 0 else end)]
    return m


def asm_memory(ctx, reset_peak=False):
    """(current, peak) device bytes held by the operator assembly of a context (include/mxasm.h: mxg_asm_memory)."""
    api = gpu_api()
    out = (C.c_int64 * 2)()
    if api.lib.mxg_asm_memory(ctx.h, out, 1 if reset_peak else 0) != 0:
        raise AssemblyError("mxg_asm_memory failed: %s" % api.lib.mxg_last_error().decode())
    return out[0], out[1]


def to_crs(dcsr, row_map, domain_map, layout=0):
    """MxCrsMatrix::fillComplete for a device-assembled operator: the rows row_map owns, ready to apply."""
    import maxwell_b200 as mx
    api = dcsr.api
    h = C.c_void_p()
    rc = api.lib.mxg_crs_create_from_dcsr(row_map.h, domain_map.h, dcsr.handle, int(layout), C.byref(h))
    if rc != 0:
        raise AssemblyError("mxg_crs_create_from_dcsr failed (%d): %s" % (rc, api.lib.mxg_last_error().decode()))
    A = mx.MxCrsMatrix(row_map, domain_map, dcsr.is_complex)
    A.h = h
    return A


# ---- example geometries of the reference (example/*.py), written against any shape factory with the method names of
# AssemblyAPI (the tests hand the same functions the oracle's factory to build the comparison geometry) ---------------
def pillbox_shape(S, radius=0.4, length=0.8):
    """example/pillbox.py:14-17 -- Cylinder(R, axis z) intersected with Slab(thickness, normal z)."""
    return S.intersection([S.cylinder(radius, (0, 0, 1), (0, 0, 0)), S.slab(length, (0, 0, 1), (0, 0, 0))])


def crabcav_shape(S, num_cells=4, cell_len=2.0 * 0.0192, cav_rad=0.04719, iris_rad=0.015, cav_rho=0.0136, iris_rho=0.00331):
    """example/crabcav.py:13-66 -- the 4-cell crab cavity as CSG: per half cell (cone & tube) | equator torus |
    (iris tube - iris torus), mirrored in z = 0, repeated along z and capped by a slab."""
    import math
    rho_sum = cav_rho + iris_rho
    rad_diff = cav_rad - iris_rad
    half2 = 0.25 * cell_len * cell_len
    diff2 = (rad_diff - rho_sum) ** 2
    cos_t = (rho_sum - rad_diff) * rho_sum
    cos_t += math.sqrt(half2 * (diff2 - rho_sum * rho_sum + half2))
    cos_t /= half2 + diff2
    theta = math.acos(cos_t)
    sin_t = math.sqrt(1 - cos_t * cos_t)
    cot_t = 1.0 / (sin_t / cos_t)
    cone_off = 0.5 * cell_len - iris_rho * sin_t + (iris_rad + iris_rho * (1.0 - cos_t)) * cot_t
    zhat, o = (0, 0, 1), (0, 0, 0)
    iris_tube = S.cylinder(iris_rad + iris_rho * (1.0 - cos_t), zhat, o)
    iris_torus = S.torus(iris_rad + iris_rho, iris_rho, zhat, (0, 0, 0.5 * cell_len))
    corr_iris_tube = S.subtract(iris_tube, iris_torus)
    cav_tube = S.cylinder(cav_rad - cav_rho * (1.0 - cos_t), zhat, o)
    cav_cone = S.cone(theta, zhat, (0, 0, cone_off))
    cav_torus = S.torus(cav_rad - cav_rho, cav_rho, zhat, o)
    pre_cav = S.intersection([cav_cone, cav_tube])
    half_cell = S.union([pre_cav, cav_torus, corr_iris_tube])
    full_cell = S.mirror(half_cell, zhat, o)
    inf_cells = S.repeat(full_cell, o, zhat, cell_len, num_cells // 2, num_cells // 2)
    caps = S.slab(float(num_cells) * cell_len, zhat, o)
    return S.intersection([caps, inf_cells])


def crabcav_grid(cell_res=10, pad=2, num_cells=4, cell_len=2.0 * 0.0192, cav_rad=0.04719):
    """example/crabcav.py:69-91: cell_res cells per cavity cell along z plus `pad` cells of metal around -> (n, origin, size)."""
    import math
    delta = cell_len / float(cell_res)
    nz = num_cells * cell_res + 2 * pad
    lz = float(nz) * delta
    nx = 2 * (int(math.ceil(cav_rad / delta)) + pad)
    lx = float(nx) * delta
    return (nx, nx, nz), (-0.5 * lx, -0.5 * lx, -0.5 * lz), (lx, lx, lz)


# eps diag [10.225, 10.225, 9.95], off-diag [yz, xz, xy] = [0.6736.., -0.6736.., -0.825] (MxProblem.cpp:501-506)
_S = 0.67360967926537398
SAPPHIRE = np.array([[10.225, -0.825, -_S], [-0.825, 10.225, _S], [-_S, _S, 9.95]])


def example_sim(ctx, workload, n, phase_shifts=None):
    """The workloads of bench.py as device simulations (set up, ready for op())."""
    api = gpu_api()
    if workload == "pillbox":
        sim = gpu_sim(ctx, n, origin=(-0.5,) * 3, size=(1.0,) * 3)
        sim.set_pec_shape(pillbox_shape(api))
    elif workload == "vacuum":
        sim = gpu_sim(ctx, n, origin=(0.0,) * 3, size=(1.0,) * 3)
    elif workload == "crabcav":
        nn, origin, size = crabcav_grid(cell_res=max(2, (n - 4) // 4))
        sim = gpu_sim(ctx, nn, origin=origin, size=size)
        sim.set_pec_shape(crabcav_shape(api))
    elif workload == "dsphmsph":      # example/dsphmsph.py: dielectric sphere (eps = 10) inside a PEC sphere
        sim = gpu_sim(ctx, n, origin=(-0.5,) * 3, size=(1.0,) * 3)
        sim.set_pec_shape(api.sphere(0.49, (0, 0, 0)))
        sim.add_dielectric(api.sphere(0.37, (0, 0, 0)), 10.0)
    elif workload == "phc":           # example/phc-sapph-r0.37.py: sapphire sphere in a periodic cell, Bloch phases
        sim = gpu_sim(ctx, n, origin=(-0.5,) * 3, size=(1.0,) * 3, phase_shifts=phase_shifts or (0.0, 0.0, 0.0))
        sim.add_dielectric(api.sphere(0.37, (0, 0, 0)), SAPPHIRE)
    else:
        raise AssemblyError("unknown workload %r" % workload)
    return sim.setup()


class EigenProblem:
    """Everything MxSolver needs for the projected eigensolve, assembled on the device: the re-discretisation hierarchy
    of MxEMSimHierarchy (MxEMSimHierarchy.cpp:37-76) for the vector and the scalar Laplacian, trilinear transfers
    (restriction = P^T / 8), divB / gradPsi / curlCurl on the fine grid and the mass diagonal dmA.

    sims: device simulations, fine to coarse. cuts(level, field, gids, num_global) -> (begin, end) selects this rank's
    rows of a field map (x-slabs); None = the whole map (one rank). Every operator, transfer and the mass diagonal is
    assembled on this rank's rows only (each chain factor on the rows its left neighbour reaches), so a rank's assembly
    memory and time shrink with the rank count; the rows are bit-identical to those of the global operators."""

    def __init__(self, ctx, sims, cuts=None, is_complex=False):
        import maxwell_b200 as mx
        self.sims = sims
        rng = {}
        for l, s in enumerate(sims):
            for f in ("bfield", "psifield"):
                if cuts is None:
                    rng[l, f] = (0, s.map_size(f)[0])
                else:
                    rng[l, f] = cuts(l, f, s.map(f), s.num_global(f))
        self.bmaps = [make_map(s, "bfield", *rng[l, "bfield"]) for l, s in enumerate(sims)]
        self.pmaps = [make_map(s, "psifield", *rng[l, "psifield"]) for l, s in enumerate(sims)]
        cx = is_complex
        self.vops = [to_crs(s.op("vecLapl", cx, rows=rng[l, "bfield"]), self.bmaps[l], self.bmaps[l]) for l, s in enumerate(sims)]
        self.sops = [to_crs(s.op("scaLapl", cx, rows=rng[l, "psifield"]), self.pmaps[l], self.pmaps[l]) for l, s in enumerate(sims)]
        self.Rb, self.Pb, self.Rp, self.Pp = [], [], [], []
        for l in range(len(sims) - 1):
            for f, maps, Rl, Pl in (("bfield", self.bmaps, self.Rb, self.Pb), ("psifield", self.pmaps, self.Rp, self.Pp)):
                p = sims[l].interpolator_from(sims[l + 1], f, cx, rows=rng[l, f])
                Pl.append(to_crs(p, maps[l], maps[l + 1]))
                del p
                r = sims[l].interpolator_transpose(sims[l + 1], f, cx, rows=rng[l + 1, f]).scale(0.125)
                Rl.append(to_crs(r, maps[l + 1], maps[l]))
        s0 = sims[0]
        b0, b1 = rng[0, "bfield"]
        self.divB = to_crs(s0.op("divB", cx, rows=rng[0, "psifield"]), self.pmaps[0], self.bmaps[0])
        self.gradPsi = to_crs(s0.op("gradPsi", cx, rows=(b0, b1)), self.bmaps[0], self.pmaps[0])
        self.curlCurl = to_crs(s0.op("curlCurl", cx, rows=(b0, b1)), self.bmaps[0], self.bmaps[0])
        fa = s0.op("dmA", False, rows=(b0, b1)).arrays()[2]
        self.m_diag = mx.MxMultiVector(self.bmaps[0], 1, cx)
        self.m_diag.from_host(fa.astype(np.complex128) if cx else fa)
        self.fracs = fa
