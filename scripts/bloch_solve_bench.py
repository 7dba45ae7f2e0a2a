"""The projected complex eigensolve of config C4 (phc: sapphire sphere in a periodic cell, example/phc-sapph-r0.37.py) at
bench.py's k-point and level sizes, device-assembled, with the plain grid transfers and with the Bloch-consistent ones
(EigenProblem(bloch_transfers=True), DESIGN.md GMG-bloch), alternating the two so that drift of the shared machine hits
both alike.

The plain variant runs the scalar hierarchy with remove_const_field as bench.py does; the Bloch variant asks
scalar_laplacian_has_constant_null_vector, which says no at a non-zero phase. Per run: seconds to the eigenpairs, LOBPCG
iterations, V-cycles, projection block-CG iterations, re-projections and the reference's residual / divergence checks;
at the end whether the two variants return the same eigenvalues (to 1e-7 relative, the solver tolerance being 1e-8).

Usage: python scripts/bloch_solve_bench.py [N] [repeats] [out.json]   (defaults: 192, 2, no file)
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import maxwell_b200 as mx  # noqa: E402
from maxwell_b200 import assembly as asm  # noqa: E402
from bench import PHC_PHASES, level_sizes  # noqa: E402


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:        # noqa: BLE001
        return "unknown (%s)" % e


def run(ctx, sizes, bloch, nev=10, block=16, tol=1e-8):
    ctx.sync()
    t0 = time.time()
    sims = [asm.example_sim(ctx, "phc", n, phase_shifts=PHC_PHASES) for n in sizes]
    ep = asm.EigenProblem(ctx, sims, is_complex=True, bloch_transfers=bloch)
    ctx.sync()
    setup_s = time.time() - t0
    rcf = asm.scalar_laplacian_has_constant_null_vector(sims[0]) if bloch else True
    del sims
    prec = mx.MxGeoMultigridPrec(ctx, ep.vops, ep.Rb, ep.Pb, smoother_sweeps=2, cycles=1)
    sprec = mx.MxGeoMultigridPrec(ctx, ep.sops, ep.Rp, ep.Pp, smoother_sweeps=1, cycles=1, remove_const_field=rcf)
    s = mx.MxSolver(ctx, ep.vops[0], m_diag=ep.m_diag, prec=prec, nev=nev, block_size=block, tol=tol, max_iters=200,
                    projection={"divB": ep.divB, "gradPsi": ep.gradPsi, "scaLapl": ep.sops[0], "sca_prec": sprec})
    ev = s.solve()
    res, div = s.check(ep.divB, A=ep.curlCurl)
    out = {"bloch_transfers": bloch, "remove_const_field": rcf, "seconds": s.seconds, "setup_s": round(setup_s, 2),
           "converged": int(s.converged), "iterations": int(s.iterations), "vcycles": int(s.apply_prec),
           "projection_cg_iterations": int(s.proj_cg_iters), "reprojections": int(s.reprojections),
           "eigenvalues": [float(e) for e in ev], "max_curlcurl_residual": float(np.max(res[:nev])),
           "max_divergence": float(np.max(div[:nev]))}
    del s, prec, sprec, ep
    return out


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 192
    repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 2
    path = sys.argv[3] if len(sys.argv) > 3 else None
    sizes = level_sizes(n, 1, "phc")
    ctx = mx.Context(0)
    run(ctx, [12, 6], True, nev=4, block=8)          # load the kernels
    runs = []
    for rep in range(repeats):
        for bloch in (False, True):
            r = run(ctx, sizes, bloch)
            r["repeat"] = rep
            runs.append(r)
            print(json.dumps({k: v for k, v in r.items() if k != "eigenvalues"}), flush=True)
    by = {b: [r for r in runs if r["bloch_transfers"] == b] for b in (False, True)}
    ev0, ev1 = np.array(by[False][0]["eigenvalues"]), np.array(by[True][0]["eigenvalues"])
    summary = {"n": n, "levels": sizes, "phases": PHC_PHASES, "gpu": gpu_info(),
               "seconds_plain": [r["seconds"] for r in by[False]], "seconds_bloch": [r["seconds"] for r in by[True]],
               "eigenvalues_plain": ev0.tolist(), "eigenvalues_bloch": ev1.tolist(),
               "eigenvalues_agree_1e-7": bool(len(ev0) == len(ev1) and np.allclose(ev0, ev1, rtol=1e-7, atol=0.0)),
               "max_rel_eigenvalue_difference": float(np.max(np.abs(ev0 - ev1) / np.abs(ev1))) if len(ev0) == len(ev1) else None,
               "runs": runs}
    print(json.dumps({k: v for k, v in summary.items() if k != "runs"}), flush=True)
    if path:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as f:
            json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
