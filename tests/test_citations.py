"""Every reference citation (file:line) in the public headers, the oracle and the design notes must point at an
existing file of the reference tree and a line range inside it. Needs a checkout of the reference sources (bauerca/maxwell),
named by the environment variable MAXWELL_REFERENCE_SRC; skipped without one."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("MAXWELL_REFERENCE_SRC", "")
CITE = re.compile(r"\b((?:src/|example/|test/)?Mx[A-Za-z0-9_]+\.(?:cpp|hpp|h)|(?:src/|example/)?[a-zA-Z0-9_\-\.]+\.py|test/AnasaziInterface\.cpp)"
                  r":(\d+)(?:-(\d+))?")


def _sources():
    out = []
    for rel in ("include/mxgpu.h", "include/mxsolver.h", "include/mx/MxTypes.hpp", "include/mx/MxLinAlg.hpp", "include/mx/MxSolver.hpp",
                "include/mxasm.h", "include/mx/MxAssembly.hpp", "maxwell_b200/csrc/mxg_yee.h", "maxwell_b200/csrc/mxg_shape.h",
                "maxwell_b200/csrc/mxg_eps.h", "maxwell_b200/csrc/mxg_asm_impl.h", "maxwell_b200/csrc/mxg_asm_api.inc",
                "maxwell_b200/csrc/mxg_asm.cu", "maxwell_b200/assembly.py",
                "oracle/mxo_geom.hpp", "oracle/mxo_sim.hpp", "oracle/mxo_ops.hpp", "oracle/oracle.py", "DESIGN.md", "INTEGRATION.md"):
        out.append(rel)
    return out


def _resolve(name):
    cands = [name] if "/" in name else ["src/" + name, "example/" + name, "test/" + name, name]
    for c in cands:
        p = os.path.join(REF, c)
        if os.path.isfile(p):
            return p
    return None


@pytest.mark.skipif(not (REF and os.path.isdir(REF)), reason="MAXWELL_REFERENCE_SRC does not name a reference checkout")
def test_reference_citations_resolve():
    checked, bad = 0, []
    lengths = {}
    for rel in _sources():
        text = open(os.path.join(ROOT, rel), errors="ignore").read()
        for m in CITE.finditer(text):
            name, lo, hi = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            path = _resolve(name)
            if path is None:
                # our own files are cited in the same style (tests/..., MxSolver.hpp of this repo): skip those
                if os.path.isfile(os.path.join(ROOT, name)) or os.path.isfile(os.path.join(ROOT, "include", "mx", os.path.basename(name))):
                    continue
                bad.append("%s: %s not found in the reference" % (rel, m.group(0)))
                continue
            if path not in lengths:
                lengths[path] = sum(1 for _ in open(path, errors="ignore"))
            if not (1 <= lo <= hi <= lengths[path]):
                bad.append("%s: %s outside 1..%d" % (rel, m.group(0), lengths[path]))
            checked += 1
    assert checked > 150, checked
    assert not bad, "\n".join(bad[:40])
