"""Device solve of the contact Newton steps on generated problems (tools/contact_problem.py): per Newton step the
local-block factorisation time and the GMRES time (CUDA events), iterations, restarts, the true relative residual and
the host synchronisations; on problems below --direct-max unknowns also the host ``spsolve`` time of the same Jacobian.
Non-convergence within ``maxiter`` is recorded, not hidden.  Writes one JSON file.

    python tools/contact_solve_bench.py --out profiles/contact_solve_b200.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = [("hex", 32, 1), ("tet", 18, 3), ("hex", 70, 1), ("tet", 38, 3)]


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                   # the measurement stands without it
        return {"gpu": "unknown", "error": str(e)}


def run_case(kind, n, planes, args):
    import torch
    import scipy.sparse.linalg as spla
    from porepy_b200 import krylov
    from tools.contact_problem import generated_contact_problem
    t0 = time.perf_counter()
    prob, _ = generated_contact_problem(n, kind, planes)
    prob.discretize()
    setup = time.perf_counter() - t0
    print(kind, n, planes, prob.num_dofs, "unknowns, set up in", round(setup, 2), "s", flush=True)
    blocks = krylov.LocalBlocks(prob.block_layout())
    steps = []

    def solver(J, rhs):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        blocks.factor(J)
        e[1].record()
        dx, info = krylov.gmres(J, rhs, precond=blocks, tol=args.tol, restart=args.restart, maxiter=args.maxiter)
        e[2].record()
        torch.cuda.synchronize()
        rec = {"factor_ms": e[0].elapsed_time(e[1]), "gmres_ms": e[1].elapsed_time(e[2]),
               **{k: info[k] for k in ("iterations", "restarts", "relres", "converged", "host_syncs")}}
        if prob.num_dofs <= args.direct_max and not steps:
            A, b = J.to_scipy().tocsc(), rhs.cpu().numpy()
            print("host spsolve of", A.shape[0], "unknowns ...", flush=True)
            t = time.perf_counter()
            ref = spla.spsolve(A, b)
            rec["host_spsolve_s"] = time.perf_counter() - t
            rec["rel_diff_to_spsolve"] = float(np.linalg.norm(dx.cpu().numpy() - ref) / np.linalg.norm(ref))
        steps.append(rec)
        print(kind, n, planes, rec, flush=True)
        return dx
    x0 = torch.zeros(prob.num_dofs, dtype=torch.float64, device="cuda")
    t = time.perf_counter()
    _, hist = prob.time_step(x0, solver, tol=1e-10, max_iterations=args.newton)
    return {"kind": kind, "n": n, "planes": planes, "unknowns": prob.num_dofs, "matrix_cells": int(prob.nc),
            "fracture_cells": int(sum(f.num_cells for f in prob.fractures)), "setup_s": setup,
            "newton_s": time.perf_counter() - t, "residuals": [h["residual"] for h in hist], "steps": steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "contact_solve_b200.json"))
    ap.add_argument("--tol", type=float, default=1e-12)
    ap.add_argument("--restart", type=int, default=100)
    ap.add_argument("--maxiter", type=int, default=2000)
    ap.add_argument("--newton", type=int, default=6, help="Newton steps per problem at most")
    ap.add_argument("--direct-max", type=int, default=101_000, help="host spsolve on problems up to this size")
    ap.add_argument("--cases", default=",".join(f"{k}:{n}:{p}" for k, n, p in CASES))
    args = ap.parse_args()
    res = {**gpu_info(), "tol": args.tol, "restart": args.restart, "maxiter": args.maxiter, "cuda_graph": False,
           "cases": []}
    for c in args.cases.split(","):
        kind, n, p = c.split(":")
        res["cases"].append(run_case(kind, int(n), int(p), args))
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps({"written": args.out}))


if __name__ == "__main__":
    main()
