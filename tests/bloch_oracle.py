"""TEST INFRASTRUCTURE ONLY -- the Bloch-consistent grid transfer on the CPU oracle (tests/cpp/bloch_oracle.cpp).

The oracle (oracle/) restates the reference, whose interpolator applies no Bloch factor. tests/cpp/bloch_oracle.cpp compiles
the oracle unchanged together with a restatement of the Bloch-consistent transfer (DESIGN.md GMG-bloch); the matrices it
returns are oracle matrices (oracle.oracle.Matrix), built from oracle simulations.
"""
import ctypes as C
import os
import subprocess

from oracle import oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        out_dir = os.path.join(HERE, "cpp", "_build")
        os.makedirs(out_dir, exist_ok=True)
        so = os.path.join(out_dir, "libbloch_oracle.so")
        src = os.path.join(HERE, "cpp", "bloch_oracle.cpp")
        deps = [src] + [os.path.join(ROOT, "oracle", f) for f in ("mxoracle.cpp", "mxo_ops.hpp", "mxo_sim.hpp", "mxo_geom.hpp")]
        if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            tmp = so + ".tmp%d" % os.getpid()
            subprocess.check_call([cxx, "-O2", "-std=c++17", "-fPIC", "-fopenmp", "-ffp-contract=off", "-Wall", "-Wno-sign-compare",
                                   "-shared", "-o", tmp, src])
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.mxb_build_bloch_interp.restype = C.c_void_p
        L.mxb_build_bloch_interp.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]
        L.mxo_last_error.restype = C.c_char_p
        _LIB = L
    return _LIB


def interpolator(sim_from, sim_to, field="bfield", is_complex=False, bloch=False):
    """orc.interpolator, and with bloch=True the transfer whose entries that wrap across a periodic face carry the Bloch
    factor of that direction (include/mxasm.h: MXG_INTERP_BLOCH)."""
    if not bloch:
        return orc.interpolator(sim_from, sim_to, field=field, is_complex=is_complex)
    orc.lib()
    h = lib().mxb_build_bloch_interp(sim_from.h, sim_to.h, field.encode(), int(is_complex))
    if not h:
        raise RuntimeError(lib().mxo_last_error().decode())
    return orc.Matrix(h)
