#!/usr/bin/env python
"""bench.py -- MPFA + MPSA interaction-region assembly throughput (3-D cells/s) and SpMV GB/s.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME]

One "step" = one full MPFA assembly (all six matrices) + one full MPSA assembly (all four matrices) of the
workload grid, inputs resident in HBM.  ``value`` = cells of the WHOLE mesh / device time (CUDA events on the
launching stream, max over ranks).

N > 1 (torchrun, one process per GPU): ONE mesh is sharded -- recursive coordinate bisection of the cells, every
rank takes the interaction regions of its own cells' nodes plus one halo layer of cells
(``porepy_b200.shard``; no data-path collective in the assembly, SURVEY.md 8e) -> strong scaling on a shared
mesh.  The sharded flow system (rows of the rank's own cells, assembled on the device from its shard only) is then
solved by the distributed Jacobi-BiCGStab (NCCL: ghost entries by point-to-point, dot products by all-reduce).

``e2e`` = the same mesh through the reference-facing operator API from HOST arrays (page-locked):
``pb.Mpfa(kw).discretize`` + ``assemble_matrix_rhs`` and ``pb.Mpsa(kw).discretize`` + ``assemble_matrix_rhs``,
with [N > 1: the shard extraction,] the topology plan, every H2D copy, the kernels, the device-side system assembly
and the D2H of the right-hand sides and of a checksum of the system values inside the timed region.  The ten
discretization matrices and the two system matrices stay in HBM behind scipy-compatible lazy matrices
(``porepy_b200.sparse.LazyCsr``); ``e2e.variants`` also reports the same call with the two system matrices, and
with all ten matrices, fetched to the host.

``--impl reference`` times the UNMODIFIED reference (``pp.Mpfa.discretize`` + ``pp.Mpsa.discretize``, loaded from
/root/reference or oracle/_ref) on the host cores, on a bounded sample of the same kind of mesh.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (kind, dims, description)
    "tet1m": ("tet", (55, 55, 55), "MPFA+MPSA assembly, structured tetrahedral grid 55^3 x 6 = 998,250 cells "
                                   "(BASELINE config[1] size; gmsh fracture meshes cannot be generated offline)"),
    "cart128": ("cart", (128, 128, 128), "MPFA+MPSA assembly, Cartesian 128^3 = 2,097,152 cells (config[2] size)"),
    "cart64": ("cart", (64, 64, 64), "MPFA+MPSA assembly, Cartesian 64^3 = 262,144 cells"),
    "cart32": ("cart", (32, 32, 32), "MPFA+MPSA assembly, Cartesian 32^3 = 32,768 cells (config[0])"),
    "tet100k": ("tet", (26, 26, 26), "MPFA+MPSA assembly, structured tetrahedral grid 26^3 x 6 = 105,456 cells"),
    "tet10k": ("tet", (12, 12, 12), "MPFA+MPSA assembly, structured tetrahedral grid 12^3 x 6 = 10,368 cells"),
    "tet384": ("tet", (4, 4, 4), "tooling: 384 tets (compute-sanitizer runs)"),
    "cart512": ("cart", (8, 8, 8), "tooling: 512 hexes (compute-sanitizer runs)"),
}
CPU_SAMPLE = {"tet": (8, 8, 8), "cart": (20, 20, 20)}   # 3,072 tets / 8,000 hexes: 10-20 s of reference time
# the value arrays one step assembles, in the order of the plan's output keys (PB_OUT_* in include/poreb200.h)
STEP_OUTPUTS = ("flux", "bound_flux", "bound_pressure_cell", "bound_pressure_face", "vector_source",
                "bound_pressure_vector_source", "stress", "bound_stress", "bound_displacement_cell",
                "bound_displacement_face")
DUMP_BYTES = 64 << 20


def make_grid(kind, dims, seed=0):
    import porepy_b200 as pb
    if kind == "tet":
        return pb.structured_tet_grid(dims)
    return pb.cart_grid_3d(dims, perturb=0.2, seed=seed)


def make_params(g, seed=0):
    import porepy_b200 as pb
    rng = np.random.default_rng(seed)
    nc = g.num_cells
    k = pb.SecondOrderTensor(1 + rng.random(nc), 1 + rng.random(nc), 1 + rng.random(nc),
                             0.3 * rng.random(nc), 0.3 * rng.random(nc), 0.3 * rng.random(nc))
    bf = g.get_all_boundary_faces()
    x = g.face_centers[0, bf]
    bc = pb.BoundaryCondition(g, bf[(x < 1e-10) | (x > 1 - 1e-10)], "dir")
    C = pb.FourthOrderTensor(np.exp(0.5 * rng.standard_normal(nc)), np.exp(0.5 * rng.standard_normal(nc)))
    vbc = pb.BoundaryConditionVectorial(g, bf[g.face_centers[2, bf] < 1e-10], "dir")
    return k, bc, C, vbc


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                    "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def gj_flops(nsf_unknowns, nrhs):
    """FP64 flops of one Gauss-Jordan solve of order n with nrhs right-hand sides."""
    n = np.asarray(nsf_unknowns, dtype=np.float64)
    w = n + nrhs
    # sum_p (n-1) * (w-p-1) multiply-adds
    return 2.0 * (n - 1) * (n * w - n * (n + 1) / 2.0)


def reference_available():
    from oracle import ref_loader
    return ref_loader.reference_available()


def reference_pass(kind, dims, seed=0, threads=None):
    """One CPU pass of the UNMODIFIED reference (``pp.Mpfa.discretize`` + ``pp.Mpsa.discretize``, loaded from
    /root/reference or oracle/_ref) on a sample grid of the workload's kind; returns (cells, s_mpfa, s_mpsa)."""
    from oracle import ref_loader
    pp = ref_loader.load_porepy()
    if threads:
        import numba
        numba.set_num_threads(min(int(threads), numba.config.NUMBA_NUM_THREADS))
    g = make_grid(kind, dims, seed)
    k, bc, C, vbc = make_params(g, seed)
    t_f, t_s, _, _ = ref_loader.reference_discretize(pp, g, k, bc, C, vbc)
    return g.num_cells, t_f, t_s


def oracle_pass(kind, dims, seed):
    """Fallback when the reference is not on the box: the NumPy restatement (oracle/fv_oracle.py)."""
    import porepy_b200 as pb
    from oracle import fv_oracle as fo
    g = make_grid(kind, dims, seed)
    k, bc, C, vbc = make_params(g, seed)
    eta = pb.determine_eta(g)
    t0 = time.perf_counter()
    fo.mpfa(g, k.values, bc, eta)
    t1 = time.perf_counter()
    fo.mpsa(g, C.values, vbc, eta)
    return g.num_cells, t1 - t0, time.perf_counter() - t1


def cpu_reference_throughput(kind, passes=1, warm=True):
    """cells/s of the reference CPU path on ONE fixed sample grid (CPU_SAMPLE), in this process.  The reference
    is single-threaded Python/SciPy except ``invert_diagonal_blocks`` (numba, all cores): ``cores`` reports the
    numba thread count.  Returns a ``cpu_baseline`` dict."""
    dims = CPU_SAMPLE[kind]
    if reference_available():
        import numba
        if warm:
            reference_pass(kind, (3, 3, 3))  # numba JIT + caches, untimed (SURVEY 8d)
        res = [reference_pass(kind, dims) for _ in range(passes)]
        cores, kind_s = numba.get_num_threads(), "reference"
        what = "pp.Mpfa.discretize + pp.Mpsa.discretize of the unmodified reference (oracle/ref_loader.py)"
    else:
        res = [oracle_pass(kind, dims, 0) for _ in range(passes)]
        cores, kind_s = 1, "port"
        what = "oracle/fv_oracle.py (reference not on this box: run oracle/make_ref.sh)"
    cells = res[0][0]
    secs = [r[1] + r[2] for r in res]
    v = cells / min(secs)
    return {"value": v, "unit": "cells/s", "cores": cores, "kind": kind_s,
            "sample": f"{what} on a {'x'.join(map(str, dims))}{' x6 tet' if kind == 'tet' else ' Cartesian'} grid "
                      f"({cells} cells), best of {passes} pass(es), numba warm-up untimed; "
                      f"seconds mpfa/mpsa of the best pass: "
                      f"{res[int(np.argmin(secs))][1]:.2f}/{res[int(np.argmin(secs))][2]:.2f}",
            "host_cpu_count": os.cpu_count(), "seconds_all_passes": secs}


def run_reference(args, rank, world):
    """``--impl reference``: the reference's own CPU implementation on the host cores (rank 0 only).  One step =
    one MPFA + MPSA discretization of the fixed sample grid of the workload's kind; the warm-up steps run the numba
    JIT on a 3^3 grid.  cells/s of the reference is size independent within ~20 % (SURVEY 8d), which is what makes
    a bounded sample of the same kind of mesh a fair denominator."""
    if rank != 0:
        return
    kind, dims, desc = WORKLOADS[args.workload]
    if reference_available():
        reference_pass(kind, (3, 3, 3))
    t_all = time.perf_counter()
    cb = cpu_reference_throughput(kind, passes=max(args.steps, 1), warm=False)
    elapsed = time.perf_counter() - t_all
    secs = cb["seconds_all_passes"]
    cells = int(np.prod(CPU_SAMPLE[kind])) * (6 if kind == "tet" else 1)
    value = float(cells / np.mean(secs))
    cb["value"] = value
    line = {
        "impl": "reference", "metric": "3D cells/sec MPFA+MPSA assembly", "value": value,
        "unit": "cells/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * elapsed / max(args.steps, 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": desc, "same_config": False,
                   "note": "same mesh generator, parameters and outputs as the GPU arm; bounded sample size "
                           f"({cells} cells per step instead of the full workload, which takes the reference "
                           "5-15 min per pass); reference cells/s is size independent within ~20 %"},
        "cpu_baseline": cb,
        "e2e": {"value": value, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))



def md_network_problem(kind, dims, n_fractures=10, aperture=1e-3, normal_permeability=1.0, seed=0):
    """BASELINE config[1]'s shape: a 3-D grid of the workload's kind cut by ``n_fractures`` disjoint planar fractures
    (``porepy_b200.mdgrid``), conductive fractures, Dirichlet pressure on two sides.  Returns the
    ``MixedDimensionalFlow`` problem and a description."""
    import porepy_b200 as pb
    from porepy_b200 import mdgrid
    from porepy_b200.mdflow import MdInterface, MdSubdomain, MixedDimensionalFlow
    g = pb.structured_tet_grid(dims) if kind == "tet" else pb.cart_grid_3d(dims)
    n = int(dims[0])
    h = 1.0 / n
    lo, hi = round(0.1 * n) * h, round(0.9 * n) * h
    planes = np.unique(np.round(np.linspace(0.08, 0.92, n_fractures) * n).astype(int))
    planes = planes[(planes > 0) & (planes < n)]
    sets = [mdgrid.faces_on_rectangle(g, 0, p * h, (lo, lo), (hi, hi)) for p in planes]
    net = mdgrid.split_fractures(g, [s for s in sets if s.size])
    m = net.matrix
    rng = np.random.default_rng(seed)
    west = np.flatnonzero(m.face_centers[0] < 1e-12)
    east = np.flatnonzero(m.face_centers[0] > 1 - 1e-12)
    bcv = np.zeros(m.num_faces)
    bcv[west] = 1.0
    k3 = pb.SecondOrderTensor(1 + rng.random(m.num_cells), 1 + rng.random(m.num_cells), 1 + rng.random(m.num_cells))
    bc3 = pb.BoundaryCondition(m)
    bc3.is_neu[west] = bc3.is_neu[east] = False
    bc3.is_dir[west] = bc3.is_dir[east] = True
    subs = [MdSubdomain(m, pb.initialize_data({}, "flow", {"second_order_tensor": k3, "bc": bc3}), bcv)]
    intfs = []
    for j, fg in enumerate(net.fractures):
        kf = pb.SecondOrderTensor(aperture * 1e4 * (1 + rng.random(fg.num_cells)))   # tangential k x specific volume
        subs.append(MdSubdomain(fg, pb.initialize_data({}, "flow", {"second_order_tensor": kf, "bc": pb.BoundaryCondition(fg),
                                                                    "ambient_dimension": 3})))
        it = net.interfaces[j]
        intfs.append(MdInterface(0, j + 1, it["mortar_to_primary_int"], it["primary_to_mortar_avg"],
                                 it["mortar_to_secondary_int"], it["secondary_to_mortar_avg"],
                                 np.full(it["cell_volumes"].size, normal_permeability), it["cell_volumes"],
                                 np.full(fg.num_cells, aperture)))
    prob = MixedDimensionalFlow(subs, intfs)
    prob.bench_extras = {"west": west, "east": east, "porosity": 0.2, "aperture": aperture}
    desc = {"matrix_cells": int(m.num_cells), "fractures": len(net.fractures),
            "fracture_cells": int(sum(f.num_cells for f in net.fractures)),
            "mortar_cells": int(sum(i.num_cells for i in intfs)), "dofs": int(prob.num_dofs),
            "aperture": aperture, "normal_permeability": normal_permeability}
    return prob, desc


def md_newton_block(prob, dt=0.05, max_iterations=4):
    """One implicit time step of COMPRESSIBLE flow on the same network (``porepy_b200.mdflow_nl``: the reference's Newton
    loop, every linearization through the device AD chain, every step solved on the pressure Schur complement)."""
    import torch
    import porepy_b200 as pb
    from porepy_b200.mdflow_nl import CompressibleMixedDimensionalFlow
    ex = prob.bench_extras
    fluid = {"compressibility": 0.05, "density": 1.0, "viscosity": 1.0, "reference_pressure": 0.0}
    storage, bcs, weights = [], [], []
    for i, s in enumerate(prob.subdomains):
        g = s.sd
        sv = 1.0 if g.dim == 3 else ex["aperture"]
        storage.append(g.cell_volumes * sv * ex["porosity"])
        bc = pb.BoundaryCondition(g)
        w = np.zeros(g.num_faces)
        if g.dim == 3:
            for f in (ex["west"], ex["east"]):
                bc.is_neu[f] = False
                bc.is_dir[f] = True
            w[ex["west"]] = fluid["density"] * np.exp(fluid["compressibility"] * 1.0) / fluid["viscosity"]   # p_b = 1
            w[ex["east"]] = fluid["density"] / fluid["viscosity"]                                             # p_b = 0
        bcs.append(bc)
        weights.append(w)
    nl = CompressibleMixedDimensionalFlow(prob.subdomains, prob.interfaces, fluid, storage, bcs, weights)
    x0 = torch.zeros(nl.num_dofs, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    x, hist = nl.time_step(x0, dt, tol=1e-8, max_iterations=max_iterations, linear_tol=1e-8)
    torch.cuda.synchronize()
    ps, lam = nl.split(x.cpu().numpy())
    return {"what": "compressible fluid (c = 0.05), storage term, upwinded mobility; Newton from p = 0, one time step",
            "dt": dt, "seconds": time.perf_counter() - t0, "history": hist,
            "pressure_range_matrix": [float(ps[0].min()), float(ps[0].max())]}


def md_network_block(kind, dims, solve=True, newton=True):
    """Mixed-dimensional flow through the operator API and the device AD chain (row g1): every subdomain by
    ``pb.Mpfa.discretize`` from host arrays, the coupled Jacobian block by block on the device (and once through the AD
    chain), then BiCGStab on the pressure Schur complement.  Wall-clock seconds with device synchronisation on both sides of every stage."""
    import torch
    t0 = time.perf_counter()
    prob, desc = md_network_problem(kind, dims)
    desc["mesh_seconds_host"] = time.perf_counter() - t0
    out = {"problem": desc, "calls": []}
    J = rhs = None
    for rep in range(3):                          # first call: plans and pools are cold
        for s in prob.subdomains:
            s.data.pop("discretization_matrices", None)
        J = rhs = None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        prob.discretize()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        J, rhs = prob.assemble()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        out["calls"].append({"discretize_s": t1 - t0, "assemble_s": t2 - t1})
    last = out["calls"][-1]
    cells = desc["matrix_cells"] + desc["fracture_cells"]
    out.update(jacobian_nnz=int(J.nnz), jacobian_rows=int(J.shape[0]),
               seconds_per_assembly=last["discretize_s"] + last["assemble_s"],
               cells_per_s=cells / (last["discretize_s"] + last["assemble_s"]),
               matrix_d2h_bytes=0,
               what="host arrays -> MPFA on the 3-D grid and every fracture plane (operator API) -> coupled Jacobian and "
                    "right-hand side resident on the device")
    ms = J.bench(20)
    out["spmv"] = {"ms": ms, "achieved_GBs": J.algorithmic_bytes() / (ms * 1e-3) / 1e9}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    Jad, _ = prob.assemble_ad()
    torch.cuda.synchronize()
    out["assemble_ad_s"] = time.perf_counter() - t0      # the reference's evaluation order (forward-mode AD chain)
    out["assemble_ad_nnz"] = int(Jad.nnz)
    del Jad
    if solve:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        x, info = prob.solve(tol=1e-8, maxiter=4000)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        res = rhs - (J @ x)
        ps, lam = prob.split(x.cpu().numpy())
        out["solve"] = {"method": info.get("method"), "preconditioner": "Jacobi on the Schur complement's diagonal",
                        "interface_block": f"{info.get('sweeps')} Jacobi sweeps per application of D^-1",
                        "tol": 1e-8, "iterations": int(info["iterations"]), "converged": bool(info["converged"]),
                        "breakdown": bool(info.get("breakdown", False)), "seconds": dt,
                        "true_relres_full_system": float(torch.linalg.vector_norm(res) / torch.linalg.vector_norm(rhs)),
                        "pressure_range_matrix": [float(ps[0].min()), float(ps[0].max())],
                        "interface_flux_abs_sum": float(sum(np.abs(v).sum() for v in lam))}
    if newton and out["assemble_ad_s"] < 5.0:
        try:
            del J, rhs
            out["newton"] = md_newton_block(prob)
        except Exception as e:     # an extra of the extra
            out["newton"] = {"error": f"{type(e).__name__}: {e}"}
    return out


def dump_outputs(out_dir, outputs):
    """Write each ``DeviceValues`` of ``outputs`` to ``out_dir/<name>.npy`` (float64), at most ``DUMP_BYTES`` in all: an
    array longer than its share is cut to a sample at seeded positions, the same in every run on the same workload, so
    that the files of two builds compare entry by entry.  The kernels add the contributions of the interaction regions
    with atomics, so two runs of one build agree in all but the last bits, not bit for bit."""
    os.makedirs(out_dir, exist_ok=True)
    cap = (DUMP_BYTES - 4096) // (8 * len(outputs))          # 4 KB for the .npy headers
    for name, vals in outputs.items():
        v = vals.download()
        if v.size > cap:
            v = v[np.sort(np.random.default_rng(0).choice(v.size, cap, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), np.array(v, dtype=np.float64))


def pinned_copy(a):
    """Page-locked copy of a host array (the e2e inputs are read by H2D copies at full PCIe rate)."""
    from porepy_b200 import _lib
    a = np.ascontiguousarray(a)
    out = _lib.pinned_empty(a.size, a.dtype).reshape(a.shape)
    out[...] = a
    return out


def pin_grid(g):
    for attr in ("nodes", "face_normals", "face_centers", "face_areas", "cell_centers", "cell_volumes"):
        setattr(g, attr, pinned_copy(np.asarray(getattr(g, attr), dtype=np.float64)))
    return g


def input_bytes(g, k, C):
    import scipy.sparse as sps
    cf, fn = sps.csc_matrix(g.cell_faces), sps.csc_matrix(g.face_nodes)
    topo = 4 * (cf.indptr.size + cf.indices.size + fn.indptr.size + fn.indices.size) + cf.nnz
    geo = 8 * (g.nodes.size + g.face_normals.size + g.face_centers.size + g.face_areas.size
               + g.cell_centers.size + g.cell_volumes.size)
    return int(topo + geo + k.values.nbytes + C.values.nbytes + 4 * g.num_faces)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("PB_BENCH_WORKLOAD", "tet1m"),
                    choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-spmv", action="store_true")
    ap.add_argument("--no-krylov", action="store_true")
    ap.add_argument("--no-mech-solve", action="store_true", help="skip the block-Jacobi solve of the mechanics system")
    ap.add_argument("--no-md-network", action="store_true", help="skip the mixed-dimensional fracture-network extra (N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the ten matrices' value arrays of the last timed step (rank 0) to DIR/<name>.npy, "
                         "float64, 64 MB in all (seeded samples of the larger arrays)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)

    # Only the JSON line may reach stdout: libraries (NCCL prints its version banner on the first
    # communicator) write to fd 1, so park fd 1 on stderr until the line is printed.
    sys.stdout.flush()
    _saved_stdout_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line: str) -> None:
        sys.stdout.flush()
        os.dup2(_saved_stdout_fd, 1)
        print(line, flush=True)
        os.dup2(2, 1)

    import torch
    import porepy_b200 as pb
    from porepy_b200 import _lib
    from porepy_b200 import krylov as kr
    from porepy_b200 import shard as sh
    from porepy_b200.sparse import LazyCsr, materialize
    lib = _lib.load()
    if lib.pb_device_count() < 1:
        raise SystemExit("bench.py: no CUDA device; porepy_b200 has no CPU path")
    _lib.check(lib.pb_set_device(local))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def allmax(vals):
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def allsum(vals):
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    # ---- ONE global mesh on every rank's host (the input of the run), sharded for N > 1
    kind, dims, desc = WORKLOADS[args.workload]
    gg = make_grid(kind, dims, seed=0)
    gk, gbc, gC, gvbc = make_params(gg, seed=0)
    nc_global = gg.num_cells
    eta = pb.determine_eta(gg)
    bv = np.zeros(gg.num_faces)
    bfaces = gg.get_all_boundary_faces()
    bv[bfaces[gg.face_centers[0, bfaces] < 1e-10]] = 1.0           # unit pressure on x = 0
    part = sh.partition_cells(gg, world) if world > 1 else None

    def my_problem():
        """This rank's grid and parameters: the whole mesh (N = 1) or its shard, from the global host arrays."""
        if world == 1:
            return None, gg, gk, gbc, gC, gvbc, bv
        s = sh.extract_shard(gg, part, rank)
        # the cell tensors stay GLOBAL: the plan restricts them on the device (DevicePlan.set_cell_map)
        return s, s.grid, gk, sh.restrict_scalar_bc(gbc, s), gC, sh.restrict_vector_bc(gvbc, s), bv[s.faces]

    shard, g, k, bc, C, vbc, bvl = my_problem()
    nc = g.num_cells
    n_own = nc if shard is None else int(shard.own_cell.sum())
    from porepy_b200.fv import scalar_bc_codes, vector_bc_codes
    t0 = time.perf_counter()
    plan = pb.DevicePlan.for_grid(g)
    if shard is not None:
        plan.set_active_nodes(shard.own_node)
        plan.set_cell_map(shard.cells, nc_global)
    plan_s = time.perf_counter() - t0
    plan.mpfa_upload(k.values, scalar_bc_codes(bc, g.num_faces), None, eta)
    codes, robw = vector_bc_codes(vbc, 3, g.num_faces)
    plan.mpsa_upload(C.values, codes, robw, eta)

    def step():
        a = plan.mpfa_assemble(True, True, True)
        b = plan.mpsa_assemble()
        return a, b

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = lib.pb_launch_count()
    t0 = time.perf_counter()
    ms_mpfa = ms_mpsa = 0.0
    for _ in range(args.steps):
        a, b = step()
        ms_mpfa += a
        ms_mpsa += b
    barrier()
    wall = time.perf_counter() - t0
    launches = lib.pb_launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    own_ms_mpfa, own_ms_mpsa = ms_mpfa, ms_mpsa
    dev_ms, wall_ms, ms_mpfa, ms_mpsa = allmax([ms_mpfa + ms_mpsa, wall * 1e3, ms_mpfa, ms_mpsa])
    ms_per_step = dev_ms / args.steps
    value = nc_global / (ms_per_step * 1e-3)
    sz = plan.sizes()
    regions_all = allsum([float((shard.own_node.sum() if shard is not None else g.num_nodes))])[0]
    cells_all = allsum([float(nc)])[0]
    # the last step's results stay in HBM, detached from the plan, and are written after the JSON line
    last_outputs = ({name: plan.take(key) for key, name in enumerate(STEP_OUTPUTS)}
                    if args.dump_outputs and rank == 0 else None)
    del plan
    if hasattr(g, "_b200_plan"):
        del g._b200_plan

    # ---- end to end through the operator API: host arrays (page-locked) in, device-resident systems + host rhs out
    pin_grid(gg)
    gk.values, gC.values = pinned_copy(gk.values), pinned_copy(gC.values)

    def e2e_call(fetch=None):
        """One cold call: [shard extraction,] topology plan, H2D, kernels, device system assembly, rhs + checksum D2H.
        fetch: None | "systems" | "all" additionally downloads the two system matrices / all ten matrices."""
        d0 = sum(LazyCsr.downloads.values())
        tm = {}
        al0 = np.zeros(4)
        lib.pb_alloc_stats(al0.ctypes.data_as(_lib._f64p))
        t_ = time.perf_counter()

        def lap(name):
            nonlocal t_
            now = time.perf_counter()
            tm[name] = now - t_
            t_ = now
        sh_, lg, lk, lbc, lC, lvbc, lbv = my_problem()
        lap("shard_extraction")
        if hasattr(lg, "_b200_plan"):
            del lg._b200_plan               # cold: plan construction is part of the call
        pl = pb.DevicePlan.for_grid(lg)
        if sh_ is not None:
            pl.set_active_nodes(sh_.own_node)
            pl.set_cell_map(sh_.cells, nc_global)
        lap("topology_plan")
        d1 = pb.initialize_data({}, "flow", {"second_order_tensor": lk, "bc": lbc, "bc_values": lbv})
        m1 = pb.Mpfa("flow")
        m1.discretize(lg, d1)
        lap("mpfa_discretize")
        A1, b1 = m1.assemble_matrix_rhs(lg, d1)
        lap("flow_system")
        d2 = pb.initialize_data({}, "mech", {"fourth_order_tensor": lC, "bc": lvbc,
                                             "bc_values": np.zeros(3 * lg.num_faces), "source": np.zeros(3 * lg.num_cells)})
        m2 = pb.Mpsa("mech")
        m2.discretize(lg, d2)
        lap("mpsa_discretize")
        A2, b2 = m2.assemble_matrix_rhs(lg, d2)
        lap("mech_system")
        chk = (A1.device_csr.checksum(), A2.device_csr.checksum())   # device reductions, 32 bytes to the host
        lap("checksums")
        if fetch in ("systems", "all"):
            materialize({"a": A1, "b": A2})
        if fetch == "all":
            materialize(d1[pb.DISCRETIZATION_MATRICES]["flow"])
            materialize(d2[pb.DISCRETIZATION_MATRICES]["mech"])
        if fetch:
            lap("fetch_to_host")
        d2h = b1.nbytes + b2.nbytes + 32 + 8 + sum(LazyCsr.downloads.values()) - d0
        al1 = np.zeros(4)
        lib.pb_alloc_stats(al1.ctypes.data_as(_lib._f64p))
        dal = al1 - al0
        timing = {"stages_s": tm, "mpfa": m1.last_timing, "mpsa": m2.last_timing,
                  "device_alloc_outside_pool": {"cudaMalloc_calls": int(dal[0]), "cudaMalloc_s": float(dal[1]),
                                                "cudaFree_calls": int(dal[2]), "cudaFree_s": float(dal[3])}}
        return (A1, b1, A2, b2, chk, sh_, lg, d1, d2), d2h, timing

    e2e_vals, d2h_step, timing = [], 0, {}
    keep = None
    for i in range(max(args.e2e_steps, 1) + 1):
        keep = None
        import gc
        gc.collect()
        barrier()
        t0 = time.perf_counter()
        keep, d2h_step, timing = e2e_call()
        barrier()
        dt = time.perf_counter() - t0
        print(f"[bench] rank {rank} e2e call {i}: {dt:.3f} s  {timing}", file=sys.stderr)
        if i > 0:                       # the first call is the warm-up (page-locked pool, CUDA context)
            e2e_vals.append(dt)
    e2e_s = allmax([sum(e2e_vals) / len(e2e_vals)])[0]
    h2d_step = input_bytes(keep[6], k, C) + bvl.nbytes + 2 * 8 * 3 * keep[6].num_faces
    h2d_all, d2h_all = allsum([float(h2d_step), float(d2h_step)])
    e2e = {"value": nc_global / e2e_s, "unit": "cells/s", "h2d_bytes_per_step": int(h2d_all),
           "d2h_bytes_per_step": int(d2h_all), "seconds_per_step": e2e_s,
           "includes": ("shard extraction + " if world > 1 else "") +
                       "topology plan + H2D from page-locked host arrays + MPFA/MPSA kernels + device-side "
                       "A = div @ flux, A = div_nd @ stress and right-hand sides + D2H of the right-hand sides and "
                       "of the checksums of both system matrices; all twelve matrices stay in HBM behind "
                       "scipy-compatible lazy matrices",
           "result_check": {"flow_system_sum_sumsq": keep[4][0], "mech_system_sum_sumsq": keep[4][1]},
           "breakdown": timing}

    # ---- distributed Jacobi-BiCGStab on the flow system assembled above (rows of the own cells, from the shard)
    krylov = None
    if not args.no_krylov:
        A1, b1 = keep[0], keep[1]
        a_dev = A1.device_csr
        diag = torch.as_tensor(a_dev.diagonal()[:n_own], dtype=torch.float64, device="cuda")
        a_dev.truncate_rows(n_own)
        if shard is not None:
            loc = kr.local_system_from_shard(keep[5], part, a_dev)
        else:
            loc = kr.LocalSystem(0, 1, np.arange(nc), np.zeros(0, np.int64), a_dev, [0], [np.zeros(0, np.int64)])
        # self-checks of the distributed operator at full size: the halo exchange delivers the global vector at the
        # shard's ghost cells, and the residual of the returned solution is recomputed with one more distributed SpMV
        op_chk = kr.DistributedOperator(loc, torch.device("cuda", local))
        cells_local = np.arange(nc) if shard is None else keep[5].cells
        probe = np.sin(0.37 * np.arange(nc_global))
        xb = op_chk.exchange(torch.as_tensor(probe[cells_local[:n_own]], device="cuda")).cpu().numpy()
        halo_err = float(np.abs(xb - probe[cells_local]).max())
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        x, info = kr.solve_local(loc, b1[:n_own], diag_own=diag, tol=1e-8, maxiter=3000)
        barrier()
        solve_s = allmax([time.perf_counter() - t0])[0]
        b_t = torch.as_tensor(b1[:n_own], device="cuda")
        res = b_t - op_chk.matvec(x)
        rr, bbn = allsum([float(res @ res), float(b_t @ b_t)])
        true_relres = float(np.sqrt(rr / bbn))
        # the same kernels on this rank's rows WITHOUT the collectives (ghost entries left at zero, local dot products,
        # 64 iterations, no convergence test): what one iteration costs in compute; the rest of ms_per_iteration is NCCL
        local_ms = None
        if world > 1:
            try:
                loc_nc = kr.LocalSystem(0, 1, loc.owned, loc.ghosts, a_dev, [0], [np.zeros(0, np.int64)])
                op_nc = kr.DistributedOperator(loc_nc, torch.device("cuda", local))
                kr.bicgstab(op_nc, b_t, tol=0.0, maxiter=16, diag_own=diag)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                _, inc = kr.bicgstab(op_nc, b_t, tol=0.0, maxiter=64, diag_own=diag)
                torch.cuda.synchronize()
                local_ms = allmax([1e3 * (time.perf_counter() - t0) / 64])[0]
                del op_nc, loc_nc
            except Exception as e:
                local_ms = f"{type(e).__name__}: {e}"
        krylov = {"system": "A = div @ flux of the sharded mesh (rows of each rank's own cells)", "rows": int(nc_global),
                  "inputs_finite": bool(np.isfinite(b1).all() and bool(torch.isfinite(diag).all())),
                  "halo_exchange_max_error": allmax([halo_err])[0], "true_relres": true_relres,
                  "cuda_graph": info.get("cuda_graph"),
                  "diag_min": float(diag.min()), "fused": bool(info.get("fused", False)),
                  "host_syncs": info.get("host_syncs"), "breakdown": info.get("breakdown"),
                  "iterations": info["iterations"], "converged": bool(info["converged"]), "relres": info["relres"],
                  "seconds": solve_s, "spmv": info["spmv"], "allreduce": info["allreduce"],
                  "halo_bytes_per_spmv_all_ranks": int(allsum([float(info["halo_bytes_per_spmv"])])[0]),
                  "ms_per_iteration": 1e3 * solve_s / max(info["iterations"], 1),
                  "ms_per_iteration_without_collectives": local_ms,
                  "nccl_share_of_iteration": (None if not isinstance(local_ms, float) else
                                              max(0.0, 1.0 - local_ms / (1e3 * solve_s / max(info["iterations"], 1)))),
                  "collectives": "ghost entries: NCCL send/recv per neighbour; dots: one all-reduce of 1-3 doubles"
                  if world > 1 else "none (single GPU)"}
        del x, loc, op_chk
        # ---- the mechanics system A = div_nd @ stress (3 x 3 blocks per cell pair) with block-Jacobi BiCGStab; N > 1: rows
        # of each rank's own cells from its shard, the halo plan with 3 unknowns per cell
        if not args.no_mech_solve:
            try:
                A2, b2 = keep[2], keep[3]
                m_dev = A2.device_csr
                barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                blk = m_dev.block_diagonal_inverse(3, nblocks=n_own)
                m_dev.truncate_rows(3 * n_own)
                if shard is not None:
                    loc2 = kr.local_system_from_shard(keep[5], part, m_dev, dof=3)
                else:
                    loc2 = kr.LocalSystem(0, 1, np.arange(3 * nc), np.zeros(0, np.int64), m_dev, [0], [np.zeros(0, np.int64)])
                cells_own = (np.arange(nc) if shard is None else keep[5].cells)[:n_own]
                body = np.random.default_rng(5).standard_normal(3 * nc_global)       # a body force, the same on every rank
                own_dofs = (cells_own[:, None] * 3 + np.arange(3)).ravel()
                rhs2 = np.asarray(b2, dtype=np.float64)[:3 * n_own] + np.repeat(np.asarray(g.cell_volumes)[:n_own], 3) * body[own_dofs]
                xm, im = kr.solve_local(loc2, rhs2, tol=1e-6, maxiter=1500, block_inv=(blk, 3))
                barrier()
                torch.cuda.synchronize()
                mech_s = allmax([time.perf_counter() - t0])[0]
                opm = kr.DistributedOperator(loc2, torch.device("cuda", local))
                rt = torch.as_tensor(rhs2, device="cuda")
                resm = rt - opm.matvec(xm)
                rrm, bbm = allsum([float(resm @ resm), float(rt @ rt)])
                krylov["mechanics"] = {
                    "system": "A = div_nd @ stress (device-assembled, 3 dof per cell), body-force right-hand side",
                    "rows": int(3 * nc_global), "nnz_rank0": int(m_dev.nnz), "preconditioner": "block Jacobi (inverted 3 x 3 cell "
                    "blocks, pb_csr_block_diag_inv_dev)", "tol": 1e-6, "iterations": im["iterations"],
                    "converged": bool(im["converged"]), "relres": im["relres"], "true_relres": float(np.sqrt(rrm / bbm)),
                    "seconds": mech_s, "ms_per_iteration": 1e3 * mech_s / max(im["iterations"], 1),
                    "cuda_graph": im.get("cuda_graph"), "allreduce": im.get("allreduce"),
                    "halo_bytes_per_spmv_all_ranks": int(allsum([float(im["halo_bytes_per_spmv"])])[0])}
                del xm, loc2, opm, blk
            except Exception as e:     # the extra must never cost the bench line
                krylov["mechanics"] = {"error": f"{type(e).__name__}: {e}"}
    keep = None

    if rank != 0:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- N = 1 extras: e2e variants with the matrices fetched to the host
    variants = None
    if world == 1:
        variants = {}
        for name, fetch in (("systems_to_host", "systems"), ("all_matrices_to_host", "all")):
            import gc
            for rep in range(2):
                gc.collect()
                t0 = time.perf_counter()
                kk, d2h_v, _ = e2e_call(fetch)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                del kk
            variants[name] = {"seconds_per_step": dt, "value": nc_global / dt, "d2h_bytes_per_step": int(d2h_v)}
        e2e["variants"] = variants

    # ---- roofline of the dominant kernel family
    plan = pb.DevicePlan.for_grid(g)
    peak, peak_src = measured_peak_hbm()
    nfc, nfb = plan.nnz(0), plan.nnz(1)
    geo_bytes = 8 * (g.nodes.size + g.face_normals.size + g.face_centers.size + g.face_areas.size
                     + g.cell_centers.size + g.cell_volumes.size)
    topo_bytes = 4 * sz["subcells"] + 4 * sz["subfaces"] + 2 * sz["subhalffaces"]
    bytes_mpfa = geo_bytes + topo_bytes + 72 * nc + g.num_faces + 8 * (2 * nfc + 2 * nfb + 6 * nfc)
    bytes_mpsa = geo_bytes + topo_bytes + 648 * nc + 3 * g.num_faces + 8 * 9 * (2 * nfc + 2 * nfb)
    dom = "mpsa" if own_ms_mpsa >= own_ms_mpfa else "mpfa"
    dom_ms = (own_ms_mpsa if dom == "mpsa" else own_ms_mpfa) / args.steps
    dom_bytes = bytes_mpsa if dom == "mpsa" else bytes_mpfa
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    # FP64 work of the local solves (Gauss-Jordan), from the plan's per-node sizes
    import scipy.sparse as sps
    fn = sps.csc_matrix(g.face_nodes)
    nsf_node = np.bincount(fn.indices, minlength=g.num_nodes)
    cn = (abs(g.face_nodes) @ abs(g.cell_faces))
    cn.data[:] = 1
    nsc_node = np.asarray(cn.sum(axis=1)).ravel()
    act = np.ones(g.num_nodes, bool) if shard is None else shard.own_node
    fl_mpfa = float(gj_flops(nsf_node[act], nsc_node[act] * 4).sum())
    fl_mpsa = float(gj_flops(3 * nsf_node[act], nsc_node[act] * 3).sum())
    fl_dom = fl_mpsa if dom == "mpsa" else fl_mpfa
    import ctypes
    fp64_peak = {}
    for kind_id, nm in ((0, "dmma_tflops"), (1, "dfma_tflops")):
        v = ctypes.c_double()
        _lib.check(lib.pb_fp64_peak(kind_id, ctypes.byref(v)))
        fp64_peak[nm] = v.value
    fp64_peak["how"] = "dependency-free register loops, 148 SMs x 8 CTAs x 256 threads, best of 5 (csrc/peaks.cu)"
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json"))).get(args.workload)
        if tj and dom in tj["kernel"] and world == 1:
            traffic = int(tj["dram_bytes_read"] + tj["dram_bytes_write"])
    except Exception:
        pass
    roofline = {
        "kernel": f"{dom}_kernel (interaction-region assembly), rank 0" + (" of its shard" if world > 1 else ""),
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": traffic, "peak_source": peak_src,
        "algorithmic_bytes_per_launch": int(dom_bytes), "ms_per_launch": dom_ms,
        "note": "latency / FP64 bound (serial pivot chain per interaction region), not HBM bound (SURVEY 8d); "
                "fp64 figures alongside",
        "fp64_gflops_achieved": fl_dom / (dom_ms * 1e-3) / 1e9,
        "fp64_peak_measured": fp64_peak,
        "fp64_frac_of_measured_dmma": (fl_dom / (dom_ms * 1e-3) / 1e12 / fp64_peak["dmma_tflops"])
        if fp64_peak.get("dmma_tflops") else None,
        "fp64_note": "Gauss-Jordan flops of the reduced local systems (from the plan's per-node sizes) over the "
                     "kernel time, against the DMMA / DFMA register-loop peaks measured in this run (pb_fp64_peak)",
        "fp64_flops_per_launch_gauss_jordan": fl_dom,
    }
    # ---- SpMV on the assembled Jacobians (HBM-bound): flow (scalar) and mechanics (3 x 3 blocks)
    spmv = None
    if not args.no_spmv:
        kk, _, _ = e2e_call()
        spmv = {}
        for name, A in (("div @ flux", kk[0]), ("div_nd @ stress", kk[2])):
            dA = A.device_csr
            ms = dA.bench(50)
            gbs = dA.algorithmic_bytes() / (ms * 1e-3) / 1e9
            spmv[name] = {"nrows": int(dA.shape[0]), "nnz": int(dA.nnz), "ms": ms, "bound": "hbm", "achieved": gbs,
                          "peak": peak, "unit": "GB/s", "frac": gbs / peak}
        del kk
    # ---- N = 1 extra: a 10-fracture mixed-dimensional network of the workload's size (BASELINE config[1])
    md = None
    if world == 1 and not args.no_md_network:
        try:
            md = md_network_block(kind, dims)
        except Exception as e:     # the extra must never cost the bench line
            md = {"error": f"{type(e).__name__}: {e}"}
    # ---- CPU baseline: the unmodified reference on a bounded sample of the same kind of mesh
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cpu = cpu_reference_throughput(kind, passes=1)
    line = {
        "metric": "3D cells/sec MPFA+MPSA assembly", "value": value, "unit": "cells/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": desc, "cells": int(nc_global), "outputs": "all six MPFA + all four MPSA matrices",
                   "l2": "inputs+outputs per step exceed the 126 MB L2 (no explicit flush)" if nc > 200000
                   else "small shard/workload: outputs of one step may fit L2",
                   "parallelism": ("single GPU" if world == 1 else
                                   f"one mesh, recursive coordinate bisection into {world} shards, node ownership + "
                                   "one halo layer of cells, no collective in the assembly"),
                   "cells_per_gpu_incl_halo": cells_all / world, "halo_cell_overhead": cells_all / nc_global - 1.0,
                   "interaction_regions_all_ranks": regions_all, "plan_seconds": plan_s,
                   "ms_mpfa": ms_mpfa / args.steps, "ms_mpsa": ms_mpsa / args.steps,
                   "wall_ms_per_step": wall_ms / args.steps},
        "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
        "spmv": spmv, "krylov": krylov, "md_network": md, "cpu_baseline": cpu,
    }
    emit(json.dumps(line))
    if last_outputs is not None:
        dump_outputs(args.dump_outputs, last_outputs)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
