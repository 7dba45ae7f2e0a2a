"""Host-side cost model that picks the dictionary SpMM kernel's thread -> row assignment
(maxwell_b200/csrc/mxg_ilv_model.h). CPU only: synthetic pattern tables in C++, and the pattern tables of real
operators from the oracle through a small extern "C" wrapper. The GPU measurements the criterion is calibrated on are
in profiles/README_r01.md; both assignments are bit-exact (tests/test_gpu_spmv.py), so a wrong choice costs time only."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
INC = os.path.join(ROOT, "maxwell_b200", "csrc")


def test_model_on_synthetic_tables(tmp_path):
    exe = str(tmp_path / "ilv_model_check")
    subprocess.check_call([CXX, "-std=c++17", "-O1", "-Wall", "-Werror", "-I", INC, os.path.join(ROOT, "tests", "cpp", "ilv_model_check.cpp"),
                           "-o", exe])
    res = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0 and "PASSED" in res.stdout, res.stdout + res.stderr


def _pattern_table(op, min_count=4):
    """(column offsets, values) dictionary of the rows, as mxg_crs_create builds it (rows seen >= min_count times)."""
    rowptr, col, val = op.arrays()
    keys, cand, row_cand = {}, [], np.empty(op.nrows, dtype=np.int64)
    for r in range(op.nrows):
        s, e = rowptr[r], rowptr[r + 1]
        d = col[s:e].astype(np.int64) - r
        k = (d.tobytes(), val[s:e].tobytes())
        i = keys.get(k)
        if i is None:
            i = keys[k] = len(cand)
            cand.append([d, 0])
        cand[i][1] += 1
        row_cand[r] = i
    keep, pat_off, delta = {}, [0], []
    for i, (d, cnt) in enumerate(cand):
        if cnt >= min_count:
            keep[i] = len(keep)
            delta.extend(d.tolist())
            pat_off.append(len(delta))
    row_pat = np.array([keep.get(i, -1) for i in row_cand], dtype=np.int32)
    return row_pat, np.array(pat_off, dtype=np.int32), np.array(delta, dtype=np.int32)


def test_model_on_real_operators(tmp_path, orc):
    so = str(tmp_path / "libilv.so")
    subprocess.check_call([CXX, "-std=c++17", "-O2", "-shared", "-fPIC", "-I", INC, os.path.join(ROOT, "tests", "cpp", "ilv_model_capi.cpp"),
                           "-o", so])
    L = C.CDLL(so)
    sim = orc.pillbox(32)
    got = {}
    for name in ("curlCurl", "vecLapl", "scaLapl", "curlE"):
        op = sim.op(name)
        rp, po, d = _pattern_table(op)
        assert (rp >= 0).mean() > 0.8
        out = (C.c_double * 5)()
        L.ilv_model_eval(rp.ctypes.data_as(C.c_void_p), po.ctypes.data_as(C.c_void_p), d.ctypes.data_as(C.c_void_p),
                         C.c_int64(0), C.c_int64(op.nrows), 8, 16, out)
        assert out[4] > 0
        got[name] = (bool(L.ilv_model_wins(out)), (out[1] + out[3]) / (out[0] + out[2]))
    # curl-curl couples the three components with component-dependent offsets: interleaving wins (measured 0.262 vs
    # 0.297 ms at 256^3); the same-offset stencils (vector / scalar Laplacian) and the curl itself keep the plain order
    assert got["curlCurl"][0] and got["curlCurl"][1] < 0.98, got
    assert not got["vecLapl"][0] and got["vecLapl"][1] > 1.3, got
    assert not got["scaLapl"][0] and not got["curlE"][0], got

