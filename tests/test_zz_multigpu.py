"""Two ranks, two GPUs, NCCL: ONE mesh is sharded, every rank assembles the rows of its own cells on its own device
from its shard only, and the distributed fused BiCGStab (ghost entries by NCCL point-to-point, dot products by
all-reduce of slices of the device scalar buffer) reproduces the direct solve of the unsplit system.  Also checks the
halo exchange itself and one distributed SpMV.  Skipped on boxes with fewer than two GPUs (the driver's single-GPU run);
run with ``gpurun --gpus 2``."""
import os

import numpy as np
import pytest
import scipy.sparse as sps
import scipy.sparse.linalg as spla

pytestmark = pytest.mark.gpu


def _ngpu():
    try:
        from porepy_b200 import _lib
        return _lib.load().pb_device_count()
    except Exception:
        return 0


def _problem():
    import porepy_b200 as pb
    g = pb.structured_tet_grid([9, 8, 7])
    rng = np.random.default_rng(3)
    nc = g.num_cells
    k = pb.SecondOrderTensor(1 + rng.random(nc), 1 + rng.random(nc), 1 + rng.random(nc),
                             0.3 * rng.random(nc), 0.3 * rng.random(nc), 0.3 * rng.random(nc))
    bf = g.get_all_boundary_faces()
    x = g.face_centers[0, bf]
    bc = pb.BoundaryCondition(g, bf[(x < 1e-10) | (x > 1 - 1e-10)], "dir")
    bv = np.zeros(g.num_faces)
    bv[bf[x < 1e-10]] = 1.0
    return g, k, bc, bv


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    import porepy_b200 as pb
    from porepy_b200 import _lib
    from porepy_b200 import krylov as kr
    from porepy_b200 import shard as sh
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    _lib.check(_lib.load().pb_set_device(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    g, k, bc, bv = _problem()
    # the unsplit system (every rank builds it on its own GPU: the reference of the checks)
    dg = pb.initialize_data({}, "flow", {"second_order_tensor": k, "bc": bc, "bc_values": bv})
    mg = pb.Mpfa("flow")
    mg.discretize(g, dg)
    Ag, bg = mg.assemble_matrix_rhs(g, dg)
    Ag = sps.csr_matrix(Ag)
    # this rank's shard
    part = sh.partition_cells(g, world)
    s = sh.extract_shard(g, part, rank)
    n_own = int(s.own_cell.sum())
    pb.DevicePlan.for_grid(s.grid).set_active_nodes(s.own_node)
    dl = pb.initialize_data({}, "flow", {
        "second_order_tensor": pb.SecondOrderTensor.from_values(s.restrict_cell_array(k.values)),
        "bc": sh.restrict_scalar_bc(bc, s), "bc_values": bv[s.faces], "mpfa_eta": pb.determine_eta(g)})
    ml = pb.Mpfa("flow")
    ml.discretize(s.grid, dl)
    a_dev, b_loc = ml.assemble_matrix_rhs_device(s.grid, dl)
    diag = a_dev.diagonal()[:n_own]
    a_dev.truncate_rows(n_own)
    loc = kr.local_system_from_shard(s, part, a_dev)
    dev = torch.device("cuda", rank)
    op = kr.DistributedOperator(loc, dev)
    # (1) halo exchange: the ghost part of xbuf holds the global vector at the shard's halo cells
    xg = np.random.default_rng(11).standard_normal(g.num_cells)
    x_own = torch.as_tensor(xg[s.cells[:n_own]], device=dev)
    xb = op.exchange(x_own).cpu().numpy()
    err_halo = float(np.abs(xb - xg[s.cells]).max())
    # (2) one distributed SpMV = the own rows of the unsplit product
    y = op.matvec(x_own).cpu().numpy()
    err_spmv = float(np.abs(y - (Ag @ xg)[s.cells[:n_own]]).max() / np.abs(Ag @ xg).max())
    # (3) fused solve; (4) eager solve (x0 given -> torch recurrence) on the same operator
    xf, info_f = kr.solve_local(loc, b_loc[:n_own], diag_own=diag, tol=1e-11, maxiter=2000)
    b_t = torch.as_tensor(b_loc[:n_own], device=dev)
    xe, info_e = kr.bicgstab(op, b_t, x0=torch.zeros_like(b_t), tol=1e-11, maxiter=2000,
                             diag_own=torch.as_tensor(diag, device=dev))
    out = [None] * world if rank == 0 else None
    dist.gather_object((s.cells[:n_own], xf.cpu().numpy(), xe.cpu().numpy(), info_f, info_e, err_halo, err_spmv), out, dst=0)
    if rank == 0:
        ref = spla.spsolve(sps.csc_matrix(Ag), bg)
        full_f, full_e = np.zeros(g.num_cells), np.zeros(g.num_cells)
        for o, a, b_, *_ in out:
            full_f[o], full_e[o] = a, b_
        q.put({"err_fused": float(np.linalg.norm(full_f - ref) / np.linalg.norm(ref)),
               "err_eager": float(np.linalg.norm(full_e - ref) / np.linalg.norm(ref)),
               "info_fused": out[0][3], "info_eager": out[0][4],
               "err_halo": max(o[5] for o in out), "err_spmv": max(o[6] for o in out)})
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(_ngpu() < 2, reason="needs two GPUs")
def test_two_gpu_sharded_assembly_halo_exchange_and_fused_solve():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 32700 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = q.get(timeout=600)
    for p in procs:
        p.join(120)
    print(res)
    assert res["err_halo"] == 0.0, res
    assert res["err_spmv"] < 1e-13, res
    assert res["info_eager"]["converged"] and res["err_eager"] < 1e-8, res
    assert res["info_fused"]["converged"] and res["err_fused"] < 1e-8, res
