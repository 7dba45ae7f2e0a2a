"""The C-ABI library loads on a CPU-only box and exports every symbol include/mxgpu.h declares."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols(header="mxgpu.h"):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mxg_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported(mx):
    syms = declared_symbols()
    assert len(syms) >= 45
    out = subprocess.check_output(["nm", "-D", "--defined-only", mx.library_path()], text=True)
    exported = set(re.findall(r" T (mxg_[a-z0-9_]+)", out))
    missing = [s for s in syms if s not in exported]
    assert not missing, "declared in mxgpu.h but not exported: %s" % missing
    L = mx.load_library()
    for s in syms:
        assert hasattr(L, s)
    assert L.mxg_version() >= 100


def test_assembly_header_symbols_are_exported(mx):
    """include/mxasm.h (operator assembly, SURVEY 8 f2 / f3) is served by the same library."""
    syms = declared_symbols("mxasm.h")
    assert len(syms) >= 38
    out = subprocess.check_output(["nm", "-D", "--defined-only", mx.library_path()], text=True)
    exported = set(re.findall(r" T (mxg_[a-z0-9_]+)", out))
    missing = [s for s in syms if s not in exported]
    assert not missing, "declared in mxasm.h but not exported: %s" % missing
    # shapes are host objects and work without a device; the simulation needs a context
    from maxwell_b200 import assembly as asm
    api = asm.gpu_api()
    s = api.intersection([api.cylinder(0.4, (0, 0, 1), (0, 0, 0)), api.slab(0.8, (0, 0, 1), (0, 0, 0))])
    assert s.func((0.0, 0.0, 0.0)) > 0 > s.func((0.0, 0.0, 0.45))
    with pytest.raises(asm.AssemblyError):
        api.sim(None, 4)


def test_no_cpu_fallback(mx):
    """Without a CUDA device the product path must fail loudly, never fall back."""
    import ctypes as C
    L = mx.load_library()
    h = C.c_void_p()
    rc = L.mxg_ctx_create(0, C.byref(h))
    if rc == 0:
        L.mxg_ctx_destroy(h)
        pytest.skip("a GPU is present")
    assert rc < 0
    assert b"no CPU fallback" in L.mxg_last_error()
    with pytest.raises(mx.MxError):
        mx.Context(0)


def test_product_never_imports_oracle():
    """oracle/ is test infrastructure: nothing under maxwell_b200/ or include/ may reference it."""
    bad = []
    for base in ("maxwell_b200", "include"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, base)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".inc", ".h", ".hpp", ".cpp")):
                    txt = open(os.path.join(dirpath, f), errors="ignore").read()
                    if re.search(r"(from|import)\s+oracle|liboracle|mxo_", txt):
                        bad.append(os.path.join(dirpath, f))
    assert not bad, bad


def test_hash_uniform_range(mx):
    import numpy as np
    v = mx.hash_uniform(12345, np.arange(100000), 0)
    assert v.min() >= -1.0 and v.max() < 1.0
    assert abs(v.mean()) < 0.01 and abs(v.std() - 1 / np.sqrt(3)) < 0.01
    assert not np.array_equal(v, mx.hash_uniform(12345, np.arange(100000), 1))


def test_solver_header_symbols_are_exported(mx):
    """libmxsolver.so exports everything include/mxsolver.h declares."""
    text = open(os.path.join(ROOT, "include", "mxsolver.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    syms = sorted(set(re.findall(r"\b(mxs_[a-z0-9_]+)\s*\(", text)))
    assert len(syms) >= 8
    S = mx.load_solver()
    for s in syms:
        assert hasattr(S, s), s


def test_eigvals_to_freqs(mx):
    """MxMagWaveOp::eigValsToFreqs (src/MxMagWaveOp.cpp:1252-1271): f = sqrt(ev + shift) c / 2 pi, or with 1/ev when
    the eigenvalue belongs to the shift-inverted operator. Pure host arithmetic, no GPU."""
    import numpy as np
    c = 299792458.0
    k2 = np.array([15.42, 21.19, 36.14, -1e-9])
    f = mx.eigvals_to_freqs(k2)
    np.testing.assert_allclose(f[:3].real, np.sqrt(k2[:3]) * c / (2 * np.pi), rtol=1e-15)
    assert np.all(f[:3].imag == 0) and f[3].real < 1e-3 and f[3].imag > 0   # slightly negative k^2 -> imaginary f
    shift = 10.0
    mu = 1.0 / (k2[:3] - shift)                                               # eigenvalues of (A - shift)^-1
    f2 = mx.eigvals_to_freqs(mu, shift=shift, invert=True)
    np.testing.assert_allclose(f2.real, f[:3].real, rtol=1e-13)
    assert mx.eigvals_to_freqs([]).shape == (0,)


def test_error_convention_without_gpu(mx):
    """Every entry point returns an int status and leaves a message in mxg_last_error / mxs_last_error (SURVEY section 8b:
    the reference prints and exit()s; the C ABI reports). Argument validation does not need a device."""
    import ctypes as C
    L = mx.load_library()
    S = mx.load_solver()
    assert L.mxg_mv_norm2(None, None) < 0 and b"NULL" in L.mxg_last_error()
    assert L.mxg_crs_apply(None, None, None) < 0 and b"mxg_crs_apply" in L.mxg_last_error()
    h = C.c_void_p()
    assert L.mxg_map_create(None, 10, None, 0, C.byref(h)) < 0
    assert L.mxg_mv_to_grid(None, 0, 0, 0, None, None) < 0
    assert L.mxg_crs_apply_host_batch(None, 1, None, None) < 0
    assert L.mxg_gmg_apply(None, None, None) < 0
    assert S.mxs_lobpcg(None, None, None, None, None, None, None, None, None, None) != 0
    assert b"NULL" in S.mxs_last_error()
    assert S.mxs_magwave_apply(None, None, None, None, None, None, None, None, 0.0, 1e-8, 1, None, None, None) != 0
    assert S.mxs_mag_to_elec(None, None, None, None, None) != 0
    assert S.mxs_eigvals_to_freqs(None, None, 3, 0.0, 0, None, None) != 0 and b"bad argument" in S.mxs_last_error()
