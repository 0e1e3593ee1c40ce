"""Row-distributed SpMV with halo exchange and a BiCGStab solve on top of it -- the "next" row
of the scope table (SURVEY.md §8f rank 1, §8e): the reference only has direct solvers
(``SolutionStrategy.solve_linear_system``, reference src/porepy/models/solution_strategy.py:830-884);
at 10^6 3-D cells those dominate the run time, and the north star asks for the Newton SpMV /
residual with NCCL used only for ghost entries and Krylov dot products.

One process per GPU.  Cells (rows and columns) are assigned to ranks by an ``owner`` array
(e.g. ``porepy_b200.shard.partition_cells``).  Every rank keeps the rows of its own cells in a
device-resident CSR (``DeviceCsr``) with columns renumbered as [own cells | ghost cells]; one SpMV =
pack + neighbour exchange of the ghost entries (``torch.distributed`` point-to-point, NCCL on GPUs)
+ the local ``csr_spmv_kernel`` on torch's current stream.  Dot products are local dots + one
all-reduce of 1-2 scalars.

The local SpMV runs through ``pb_csr_spmv_dev`` on raw device pointers of torch tensors (torch is
plumbing: memory + collectives).  For the CPU (gloo) tests of the host logic a ``matvec`` stand-in
can be injected; the product default has no CPU path.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
import scipy.sparse as sps


@dataclass
class LocalSystem:
    """This rank's rows of a row-distributed matrix."""

    rank: int
    world: int
    owned: np.ndarray            # global ids of own cells (ascending)
    ghosts: np.ndarray           # global ids of ghost columns, grouped by owner rank
    a_local: sps.csr_matrix      # (n_own, n_own + n_ghost), local column numbering
    recv_counts: list            # ghosts received from each rank
    send_index: list             # per rank: local indices (into own) to send
    extra: dict = field(default_factory=dict)


def build_local_system(a, owner: np.ndarray, rank: int, world: int, group=None) -> LocalSystem:
    """Split ``a`` (global scipy CSR, same on every rank) by rows; collective (exchanges the ghost lists)."""
    a = sps.csr_matrix(a)
    owner = np.asarray(owner)
    owned = np.flatnonzero(owner == rank)
    rows = a[owned]
    cols = np.unique(rows.indices)
    gh = cols[owner[cols] != rank]
    gh = gh[np.lexsort((gh, owner[gh]))]  # grouped by owner, ascending inside
    n_own = owned.size
    g2l = np.full(a.shape[1], -1, dtype=np.int64)
    g2l[owned] = np.arange(n_own)
    g2l[gh] = n_own + np.arange(gh.size)
    a_local = sps.csr_matrix((rows.data, g2l[rows.indices], rows.indptr), shape=(n_own, n_own + gh.size))
    a_local.sort_indices()
    need = [gh[owner[gh] == q] for q in range(world)]  # what I need from q
    recv_counts = [int(x.size) for x in need]
    if world > 1:
        import torch.distributed as dist
        all_need = [None] * world
        dist.all_gather_object(all_need, [x.tolist() for x in need], group=group)
        send_index = [g2l[np.asarray(all_need[q][rank], dtype=np.int64)] for q in range(world)]
    else:
        send_index = [np.zeros(0, dtype=np.int64)]
    return LocalSystem(rank, world, owned, gh, a_local, recv_counts, send_index)


def local_system_from_shard(shard, part: np.ndarray, a_rows, group=None, dof: int = 1) -> LocalSystem:
    """This rank's rows of the global system, straight from its shard (``shard.extract_shard`` numbers the own
    cells first): ``a_rows`` holds the rows of the own cells with columns in the shard's local cell numbering,
    i.e. already [own | ghost] -- a scipy CSR or a ``DeviceCsr`` (e.g. ``DevicePlan.mpfa_system()`` after
    ``truncate_rows(n_own)``).  No global matrix exists anywhere.  The ghost cells are regrouped by owner rank for
    the exchange through a column permutation of the ghost block, which is returned in ``extra["ghost_perm"]``
    and applied to the receive buffer instead of to the matrix.  ``dof`` unknowns per cell (3 for the mechanics
    system ``div_nd @ stress``: row / column ``cell * dof + component``): the cell-level halo plan is expanded.
    Collective (exchanges the ghost lists)."""
    rank = shard.rank
    part = np.asarray(part)
    n_own = int(shard.own_cell.sum())
    assert shard.own_cell[:n_own].all() and not shard.own_cell[n_own:].any(), "shard cells must be own-first"
    owned = shard.cells[:n_own]
    ghosts = shard.cells[n_own:]                      # local column n_own + i  <->  global cell ghosts[i]
    gowner = part[ghosts]
    world = 1
    if group is not None or _dist_initialized():
        import torch.distributed as dist
        world = dist.get_world_size(group)
    order = np.lexsort((ghosts, gowner))              # receive order: grouped by owner, ascending global id
    recv_counts = [int((gowner == q).sum()) for q in range(world)]
    if world > 1:
        import torch.distributed as dist
        need = [ghosts[order][gowner[order] == q].tolist() for q in range(world)]
        all_need = [None] * world
        dist.all_gather_object(all_need, need, group=group)
        g2l = {int(c): i for i, c in enumerate(owned)} if n_own < 2_000_000 else None
        lut = np.full(int(shard.num_global[0]), -1, dtype=np.int64)
        lut[owned] = np.arange(n_own)
        send_index = [lut[np.asarray(all_need[q][rank], dtype=np.int64)] for q in range(world)]
        del g2l
        for ix in send_index:
            assert (ix >= 0).all(), "a rank asked for a cell this rank does not own"
    else:
        send_index = [np.zeros(0, dtype=np.int64)]
    # position in the receive buffer of each ghost column: recv slot j holds ghost order[j]
    slot_of_ghost = np.empty(ghosts.size, dtype=np.int64)
    slot_of_ghost[order] = np.arange(ghosts.size)
    ghosts_sorted = ghosts[order]
    if dof > 1:
        ex = lambda ix: (np.asarray(ix, dtype=np.int64)[:, None] * dof + np.arange(dof)).ravel()  # noqa: E731
        owned, ghosts_sorted, slot_of_ghost = ex(owned), ex(ghosts_sorted), ex(slot_of_ghost)
        send_index = [ex(ix) for ix in send_index]
        recv_counts = [c * dof for c in recv_counts]
    return LocalSystem(rank, world, owned, ghosts_sorted, a_rows, recv_counts, send_index,
                       extra={"ghost_perm": slot_of_ghost, "dof": dof})


def _dist_initialized() -> bool:
    try:
        import torch.distributed as dist
        return dist.is_available() and dist.is_initialized()
    except Exception:
        return False


class DistributedOperator:
    """y_own = (A x)_own with x distributed; torch tensors (cuda float64; cpu only with a stand-in)."""

    def __init__(self, loc: LocalSystem, device, matvec=None, group=None):
        import torch
        self.torch = torch
        self.loc, self.device, self.group = loc, device, group
        self.n_own = loc.owned.size
        self.n_ghost = loc.ghosts.size
        self.xbuf = torch.zeros(self.n_own + self.n_ghost, dtype=torch.float64, device=device)
        self.send_idx = [torch.as_tensor(ix, dtype=torch.int64, device=device) for ix in loc.send_index]
        self.halo_bytes = 8 * sum(int(ix.numel()) for ix in self.send_idx)
        # shards keep their own ghost column order: receive into a staging buffer, then permute
        perm = loc.extra.get("ghost_perm") if loc.extra else None
        self.ghost_perm = None if perm is None else torch.as_tensor(perm, dtype=torch.int64, device=device)
        self.recv = torch.zeros(self.n_ghost, dtype=torch.float64, device=device) if perm is not None else None
        if matvec is not None:
            self._matvec = matvec  # test stand-in (host logic checks under gloo)
            self.dev_csr = None
        else:
            if torch.device(device).type != "cuda":
                raise RuntimeError("porepy_b200.krylov: the SpMV kernel needs a CUDA device (no CPU path)")
            from .sparse import DeviceCsr
            self.dev_csr = loc.a_local if isinstance(loc.a_local, DeviceCsr) else DeviceCsr(loc.a_local)
            self._matvec = None

    def exchange(self, x_own):
        """Fill xbuf = [x_own | ghosts] (neighbour exchange of the ghost entries)."""
        torch = self.torch
        self.xbuf[: self.n_own].copy_(x_own)
        if self.loc.world == 1:
            return self.xbuf
        import torch.distributed as dist
        target = self.xbuf[self.n_own:] if self.recv is None else self.recv
        ops, off = [], 0
        sends = []
        for q in range(self.loc.world):
            if q == self.loc.rank:
                continue
            if self.send_idx[q].numel():
                buf = x_own.index_select(0, self.send_idx[q]).contiguous()
                sends.append(buf)
                ops.append(dist.P2POp(dist.isend, buf, q, group=self.group))
        for q in range(self.loc.world):
            cnt = self.loc.recv_counts[q]
            if q != self.loc.rank and cnt:
                ops.append(dist.P2POp(dist.irecv, target[off:off + cnt], q, group=self.group))
            off += cnt
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()
        if self.recv is not None:
            torch.index_select(self.recv, 0, self.ghost_perm, out=self.xbuf[self.n_own:])
        return self.xbuf

    def exchange_into(self, xbuf):
        """Ghost exchange for a caller-owned buffer [x_own | ghosts] whose own part is already in place (the fused
        Krylov kernels write their output vectors straight into such buffers: no staging copy)."""
        if self.loc.world == 1:
            return xbuf
        torch = self.torch
        import torch.distributed as dist
        x_own = xbuf[: self.n_own]
        target = xbuf[self.n_own:] if self.recv is None else self.recv
        ops, off, sends = [], 0, []
        for q in range(self.loc.world):
            if q != self.loc.rank and self.send_idx[q].numel():
                buf = x_own.index_select(0, self.send_idx[q])
                sends.append(buf)
                ops.append(dist.P2POp(dist.isend, buf, q, group=self.group))
        for q in range(self.loc.world):
            cnt = self.loc.recv_counts[q]
            if q != self.loc.rank and cnt:
                ops.append(dist.P2POp(dist.irecv, target[off:off + cnt], q, group=self.group))
            off += cnt
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()
        if self.recv is not None:
            torch.index_select(self.recv, 0, self.ghost_perm, out=xbuf[self.n_own:])
        return xbuf

    def matvec(self, x_own, out=None):
        torch = self.torch
        xb = self.exchange(x_own)
        if out is None:
            out = torch.empty(self.n_own, dtype=torch.float64, device=self.device)
        if self._matvec is not None:
            out.copy_(self._matvec(xb))
        else:
            stream = torch.cuda.current_stream().cuda_stream
            self.dev_csr.spmv_device(xb.data_ptr(), out.data_ptr(), stream)
        return out

    def dots(self, pairs):
        """Global dot products of several (a, b) pairs with ONE all-reduce."""
        torch = self.torch
        v = torch.stack([torch.dot(a, b) for a, b in pairs])
        if self.loc.world > 1:
            import torch.distributed as dist
            dist.all_reduce(v, group=self.group)
        return v


def bicgstab(op: DistributedOperator, b_own, x0=None, tol: float = 1e-10, maxiter: int = 2000,
             diag_own=None, check_every: int = 8, block_inv=None):
    """Right-preconditioned BiCGStab on the distributed operator.  Preconditioner: Jacobi (``diag_own``: the diagonal of
    the own rows) or block Jacobi (``block_inv = (minv, bs)``: the inverted bs x bs diagonal blocks of the own rows as a
    flat tensor, e.g. ``DeviceCsr.block_diagonal_inverse`` -- the displacement components of a cell in the mechanics
    system), or none.
    Returns (x_own, info) with info = {"iterations", "relres", "converged", "breakdown", "spmv", "allreduce"}.
    On a CUDA operator the fused device loop runs (``_bicgstab_fused``: no host synchronisation inside the
    iteration); the eager torch recurrence below serves the CPU stand-in tests of the host logic."""
    if op.dev_csr is not None and x0 is None:
        return _bicgstab_fused(op, b_own, tol, maxiter, diag_own, check_every, block_inv)
    torch = op.torch
    x = torch.zeros_like(b_own) if x0 is None else x0.clone()
    if block_inv is not None:
        blk = block_inv[0].reshape(-1, int(block_inv[1]), int(block_inv[1]))
        prec = lambda vec: torch.bmm(blk, vec.reshape(-1, blk.shape[1], 1)).reshape(-1)  # noqa: E731
    elif diag_own is not None:
        minv = 1.0 / diag_own
        prec = lambda vec: vec * minv  # noqa: E731
    else:
        prec = lambda vec: vec  # noqa: E731
    r = b_own - op.matvec(x) if x0 is not None else b_own.clone()
    rhat = r.clone()
    bnorm = float(torch.sqrt(op.dots([(b_own, b_own)])[0]))
    if bnorm == 0.0:
        return x, {"iterations": 0, "relres": 0.0, "converged": True, "breakdown": False, "spmv": 0, "allreduce": 1}
    rho = alpha = omega = 1.0
    v = torch.zeros_like(r)
    p = torch.zeros_like(r)
    nspmv, nred, relres = 0, 1, 1.0

    def done(it, breakdown):
        return x, {"iterations": it, "relres": relres, "converged": relres < tol, "breakdown": breakdown,
                   "spmv": nspmv, "allreduce": nred}
    for it in range(1, maxiter + 1):
        # every scalar below comes out of an all-reduce: identical on all ranks, so all ranks leave together
        rho_new = float(op.dots([(rhat, r)])[0])
        nred += 1
        if rho_new == 0.0 or not np.isfinite(rho_new):
            return done(it - 1, True)
        beta = (rho_new / rho) * (alpha / omega)
        p = r + beta * (p - omega * v)
        ph = prec(p)
        v = op.matvec(ph)
        nspmv += 1
        rv = float(op.dots([(rhat, v)])[0])
        nred += 1
        if rv == 0.0 or not np.isfinite(rv):
            return done(it - 1, True)
        alpha = rho_new / rv
        s = r - alpha * v
        sh = prec(s)
        t = op.matvec(sh)
        nspmv += 1
        d = op.dots([(t, s), (t, t), (s, s)])
        nred += 1
        tt = float(d[1])
        omega = float(d[0]) / tt if tt > 0 else 0.0
        x = x + alpha * ph + omega * sh
        r = s - omega * t
        rho = rho_new
        relres = float(torch.sqrt(op.dots([(r, r)])[0])) / bnorm
        nred += 1
        if not np.isfinite(relres):
            return done(it, True)
        if relres < tol:
            return done(it, False)
        if omega == 0.0:
            return done(it, True)
    return done(maxiter, False)


def _bicgstab_fused(op: DistributedOperator, b_own, tol, maxiter, diag_own, check_every, block_inv=None):
    """The iteration on the device: three fused vector kernels (csrc/krylov.cu) and two SpMVs whose epilogue
    accumulates the dot products; all scalars of the recurrence stay in a 14-double device buffer, all-reduced in
    contiguous slices (NCCL on the same stream) under torch.distributed.  The preconditioned vectors are written
    straight into the [own | ghost] SpMV input buffers.  A block of ``check_every`` iterations is captured once in a
    CUDA graph and replayed (``POREB200_KRYLOV_GRAPH=0`` or a failed capture: plain launches); the host reads the scalar
    buffer once per block only, and a sticky device-side DONE flag freezes the vectors once the residual is below the
    tolerance, so running to the end of a block past convergence is harmless."""
    import ctypes as C
    import os
    from . import _lib
    torch = op.torch
    lib = _lib.load()
    n, ng = op.n_own, op.n_ghost
    dev = b_own.device
    world = op.loc.world
    vec = lambda m=n: torch.zeros(m, dtype=torch.float64, device=dev)  # noqa: E731
    x, r, rhat, p, v, s, t = (vec() for _ in range(7))
    xb_p, xb_s = vec(n + ng), vec(n + ng)            # SpMV inputs [own | ghost]; ph / sh are their own parts
    ph, sh = xb_p[:n], xb_s[:n]
    minv = None if diag_own is None else (1.0 / diag_own).contiguous()
    bs = 1
    if block_inv is not None:
        minv, bs = block_inv[0].contiguous(), int(block_inv[1])
        if n % bs or minv.numel() != n * bs:
            raise ValueError("block_inv: expected (n / bs) inverted bs x bs blocks of the own rows")
    scal = torch.zeros(14, dtype=torch.float64, device=dev)
    P = lambda a: C.c_void_p(a.data_ptr()) if a is not None else None  # noqa: E731
    S = lambda i: C.c_void_p(scal.data_ptr() + 8 * i)  # noqa: E731
    b_own = b_own.contiguous()
    csr = op.dev_csr
    carry = 1 if op.loc.rank == 0 else 0
    nred = [0]

    dbg_reduce = os.environ.get("POREB200_KRY_REDUCE", "")
    dbg_exch = os.environ.get("POREB200_KRY_EXCH", "")

    def reduce(lo, hi):
        if world > 1:
            import torch.distributed as dist
            if dbg_reduce == "clone":
                tmp = scal[lo:hi].clone()
                dist.all_reduce(tmp, group=op.group)
                scal[lo:hi].copy_(tmp)
            else:
                dist.all_reduce(scal[lo:hi], group=op.group)
            nred[0] += 1

    def exch(buf):
        if dbg_exch == "copy" and world > 1:
            buf.copy_(op.exchange(buf[:n].clone()))
        else:
            op.exchange_into(buf)

    def iterations(count, it0):
        stream = torch.cuda.current_stream().cuda_stream
        for it in range(it0, it0 + count):
            cur = it & 1
            g = 5 * cur
            _lib.check(lib.pb_kry_p(n, P(r), P(p), P(v), P(minv), P(ph), P(scal), cur, bs, stream))
            exch(xb_p)
            _lib.check(lib.pb_csr_spmv_dots_dev(csr.h, P(xb_p), P(v), P(rhat), S(g + 0), None, None, stream))
            reduce(g + 0, g + 1)
            _lib.check(lib.pb_kry_s(n, P(r), P(v), P(minv), P(s), P(sh), P(scal), cur, bs, stream))
            exch(xb_s)
            _lib.check(lib.pb_csr_spmv_dots_dev(csr.h, P(xb_s), P(t), P(s), S(g + 1), None, S(g + 2), stream))
            reduce(g + 1, g + 3)
            _lib.check(lib.pb_kry_xr(n, P(x), P(ph), P(sh), P(s), P(t), P(r), P(rhat), P(scal), cur, carry, stream))
            nx = 5 * (cur ^ 1)
            reduce(nx + 3, nx + 5)

    stream0 = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.pb_kry_init(n, P(b_own), P(x), P(r), P(rhat), P(p), P(v), P(scal), float(tol), stream0))
    reduce(10, 11)
    _lib.check(lib.pb_kry_seed(P(scal), stream0))
    h = scal.cpu().numpy()
    if h[10] == 0.0:
        return x, {"iterations": 0, "relres": 0.0, "converged": True, "breakdown": False, "spmv": 0, "allreduce": nred[0]}
    bb = float(h[10])
    check_every = max(2, check_every + (check_every & 1))         # even: a block starts at parity 0
    graph = None
    if os.environ.get("POREB200_KRYLOV_GRAPH", "1") != "0" and maxiter >= check_every:
        try:
            torch.cuda.synchronize()
            side = torch.cuda.Stream(device=dev)
            g_ = torch.cuda.CUDAGraph()
            red0 = nred[0]
            with torch.cuda.graph(g_, stream=side):
                iterations(check_every, 0)
            nred[0] = red0
            graph = g_
        except Exception as e:                                   # capture not possible here: plain launches
            import logging
            logging.getLogger(__name__).info("BiCGStab: CUDA graph capture failed (%s); plain launches", e)
            graph = None
            torch.cuda.synchronize()
            # a failed capture may have run nothing or a part: restart the recurrence from a clean state
            _lib.check(lib.pb_kry_init(n, P(b_own), P(x), P(r), P(rhat), P(p), P(v), P(scal), float(tol), stream0))
            reduce(10, 11)
            _lib.check(lib.pb_kry_seed(P(scal), stream0))
    it, nspmv = 0, 0
    relres, converged, breakdown = 1.0, False, False
    per_block_red = 3 if world > 1 else 0
    trace = [] if os.environ.get("POREB200_KRYLOV_TRACE") else None
    while it < maxiter:
        count = min(check_every, maxiter - it)
        if graph is not None and count == check_every:
            graph.replay()
            nred[0] += per_block_red * count
        else:
            iterations(count, it)
        it += count
        nspmv += 2 * count
        h = scal.cpu().numpy()            # the only host synchronisation: once per block
        rr = float(h[5 * (it & 1) + 3])
        if not np.isfinite(h).all():
            breakdown = True
            break
        relres = float(np.sqrt(max(rr, 0.0) / bb))
        if trace is not None:
            trace.append((it, relres) + tuple(float(v) for v in h[:10]))
        if relres <= tol:
            converged = True
            break
    done_it = int(h[12]) if np.isfinite(h[12]) else it
    return x, {"iterations": done_it if converged else it, "relres": relres, "converged": converged,
               "breakdown": breakdown, "spmv": nspmv, "allreduce": nred[0], "fused": True,
               "cuda_graph": graph is not None, "host_syncs": (it + check_every - 1) // check_every + 1,
               **({"trace": trace} if trace is not None else {})}


def solve(a, b, owner=None, tol: float = 1e-10, maxiter: int = 2000, jacobi: bool = True, device=None,
          matvec_factory=None):
    """Solve A x = b.  Single process: everything on cuda:0.  Under torch.distributed: ``a``/``b`` are
    the global system on every rank, ``owner`` assigns cells to ranks; returns the OWN part of x,
    the own global ids and the solver info."""
    import torch
    rank, world = 0, 1
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            rank, world = dist.get_rank(), dist.get_world_size()
    except Exception:
        pass
    a = sps.csr_matrix(a)
    if owner is None:
        owner = np.zeros(a.shape[0], dtype=np.int64)
        if world > 1:
            owner = (np.arange(a.shape[0]) * world) // a.shape[0]
    loc = build_local_system(a, owner, rank, world)
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else "cpu"
    mv = None if matvec_factory is None else matvec_factory(loc)
    op = DistributedOperator(loc, device, matvec=mv)
    b_own = torch.as_tensor(np.asarray(b)[loc.owned], dtype=torch.float64, device=device)
    diag = None
    if jacobi:
        dg = a.diagonal()[loc.owned]
        if np.all(dg != 0):
            diag = torch.as_tensor(dg, dtype=torch.float64, device=device)
    x, info = bicgstab(op, b_own, tol=tol, maxiter=maxiter, diag_own=diag)
    info["halo_bytes_per_spmv"] = op.halo_bytes
    return x, loc.owned, info


def solve_local(loc: LocalSystem, b_own, diag_own=None, tol: float = 1e-10, maxiter: int = 2000, device=None,
                matvec_factory=None, group=None, block_inv=None):
    """BiCGStab on a row-distributed system given by this rank's ``LocalSystem`` (e.g. from
    ``local_system_from_shard``); ``b_own`` / ``diag_own``: NumPy arrays or torch tensors of the own rows.
    Returns (x_own, info)."""
    import torch
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else "cpu"
    mv = None if matvec_factory is None else matvec_factory(loc)
    op = DistributedOperator(loc, device, matvec=mv, group=group)
    b = torch.as_tensor(np.asarray(b_own) if not torch.is_tensor(b_own) else b_own, dtype=torch.float64, device=device)
    dg = None
    if diag_own is not None:
        dg = torch.as_tensor(np.asarray(diag_own) if not torch.is_tensor(diag_own) else diag_own,
                             dtype=torch.float64, device=device)
    x, info = bicgstab(op, b, tol=tol, maxiter=maxiter, diag_own=dg, block_inv=block_inv)
    info["halo_bytes_per_spmv"] = op.halo_bytes
    return x, info


# ------------------------------------------------------------------------------------------
# restarted GMRES with a local-block preconditioner: the Newton steps of the contact models
# ------------------------------------------------------------------------------------------


def _size_classes(sizes: np.ndarray):
    """Block ids grouped by team size (s <= 4, 8, 16, 32) and the five group boundaries."""
    cls = np.searchsorted(np.array([4, 8, 16, 32]), sizes)           # 0..3 (sizes <= 32 checked by the caller)
    order = np.argsort(cls, kind="stable").astype(np.int32)
    ptr = np.concatenate(([0], np.cumsum(np.bincount(cls, minlength=4)))).astype(np.int64)
    return order, ptr


def check_block_layout(layout, n: int | None = None) -> None:
    """A layout (``ptr``, ``rows``, ``cols``) must pair every row and every column of an n x n matrix with exactly one
    block, and no block may be wider than 32."""
    ptr, rows, cols = np.asarray(layout.ptr), np.asarray(layout.rows), np.asarray(layout.cols)
    n = int(rows.size) if n is None else int(n)
    sizes = np.diff(ptr)
    if ptr[0] != 0 or ptr[-1] != rows.size or rows.size != cols.size or np.any(sizes < 1) or np.any(sizes > 32):
        raise ValueError("block layout: blocks of 1..32 rows and as many columns are expected")
    for name, ix in (("rows", rows), ("cols", cols)):
        if ix.size != n or not np.array_equal(np.bincount(ix, minlength=n), np.ones(n, np.int64)):
            raise ValueError(f"block layout: the {name} are not a bijection onto 0..{n - 1}")


class LocalBlocks:
    """Local-block inverse preconditioner (csrc/local_blocks.cu) on a fixed layout: ``layout.ptr`` (block pointers),
    ``layout.rows`` / ``layout.cols`` (row and column of every block entry; each a bijection).  The layout is uploaded
    once; ``factor(J)`` inverts the blocks ``J[rows_b, cols_b]`` of a device matrix (every Newton step), ``apply(r, out)``
    writes ``out[cols_b] = B_b^-1 r[rows_b]``.  A singular block raises ``ValueError`` naming it; there is no fallback."""

    def __init__(self, layout, device=None):
        import torch
        self.torch = torch
        check_block_layout(layout)
        ptr = np.asarray(layout.ptr, np.int64)
        sizes = np.diff(ptr)
        self.n, self.num_blocks = int(ptr[-1]), int(sizes.size)
        self.sizes = sizes
        order, self.class_ptr = _size_classes(sizes)
        inv_ptr = np.concatenate(([0], np.cumsum(sizes * sizes))).astype(np.int64)
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("porepy_b200.krylov.LocalBlocks: the block kernels need a CUDA device (no CPU path)")
        up = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)  # noqa: E731
        self.ptr, self.inv_ptr = up(ptr, torch.int64), up(inv_ptr, torch.int64)
        self.rows, self.cols = up(layout.rows, torch.int32), up(layout.cols, torch.int32)
        self.order = up(order, torch.int32)
        self.inv = torch.empty(int(inv_ptr[-1]), dtype=torch.float64, device=dev)
        self.err = torch.zeros(1, dtype=torch.int64, device=dev)
        self.device = dev

    def _args(self):
        import ctypes as C
        P = lambda a: C.c_void_p(a.data_ptr())  # noqa: E731
        return (self.num_blocks, P(self.ptr), P(self.rows), P(self.cols), P(self.inv_ptr), P(self.order),
                self.class_ptr.ctypes.data_as(C.POINTER(C.c_int64)))

    def factor(self, J, stream: int = 0) -> "LocalBlocks":
        import ctypes as C
        from . import _lib
        if tuple(J.shape) != (self.n, self.n):
            raise ValueError(f"LocalBlocks.factor: a {self.n} x {self.n} matrix is expected, got {J.shape}")
        st = stream or self.torch.cuda.current_stream().cuda_stream
        _lib.check(_lib.load().pb_csr_local_block_inv_dev(J.h, *self._args(), C.c_void_p(self.inv.data_ptr()),
                                                          C.c_void_p(self.err.data_ptr()), st))
        return self

    def apply(self, r, out=None, stream: int = 0, skip=None):
        """``skip``: a device address (int) of a double; when it holds a non-zero value the call does nothing (the
        GMRES loop passes its sticky DONE flag)."""
        import ctypes as C
        from . import _lib
        if out is None:
            out = self.torch.empty(self.n, dtype=self.torch.float64, device=self.device)
        st = stream or self.torch.cuda.current_stream().cuda_stream
        _lib.check(_lib.load().pb_local_block_apply_dev(*self._args(), C.c_void_p(self.inv.data_ptr()),
                                                        C.c_void_p(r.data_ptr()), C.c_void_p(out.data_ptr()),
                                                        None if skip is None else C.c_void_p(skip), st))
        return out


def _matvec_of(a):
    if hasattr(a, "matvec"):
        return a.matvec
    return lambda v: a @ v


def gmres(a, b, precond=None, x0=None, tol: float = 1e-12, restart: int = 100, maxiter: int = 2000,
          check_every: int = 8):
    """Restarted right-preconditioned GMRES(m) with classical Gram-Schmidt and one reorthogonalisation pass (CGS2).
    ``a``: ``DeviceCsr`` or an operator with ``matvec``; ``b``: a tensor; ``precond``: an object with
    ``apply(r, out)`` (``LocalBlocks``) or None.  Single process.  Returns (x, info), info = {"iterations" (Arnoldi
    steps), "restarts", "relres" (the TRUE residual ||b - A x|| / ||b||, recomputed at every restart and before
    convergence is reported), "converged" (relres <= tol), "host_syncs"}.
    With a ``DeviceCsr`` the device loop runs (``_gmres_fused``: all scalars on the device, one host read per
    ``check_every`` steps and one per restart); it takes a ``LocalBlocks`` preconditioner or none, any other raises
    ``TypeError``.  Otherwise the eager torch recurrence below runs, the same algorithm, which the CPU tests run on a
    matvec stand-in; it reads the Hessenberg column once per step, so its ``host_syncs`` is one per step plus one per
    restart (and one for ||b||)."""
    from .sparse import DeviceCsr
    if isinstance(a, DeviceCsr):
        if precond is not None and not isinstance(precond, LocalBlocks):
            raise TypeError("gmres: the device loop takes a krylov.LocalBlocks preconditioner or none, "
                            f"not {type(precond).__name__}")
        return _gmres_fused(a, b, precond, x0, tol, restart, maxiter, check_every)
    import torch
    mv = _matvec_of(a)
    n = b.numel()
    m = max(1, min(int(restart), n))
    x = torch.zeros_like(b) if x0 is None else x0.clone()
    bnorm = float(torch.linalg.vector_norm(b))
    syncs = 1
    if bnorm == 0.0:
        return torch.zeros_like(b), {"iterations": 0, "restarts": 0, "relres": 0.0, "converged": True, "host_syncs": syncs}
    prec = (lambda v: v) if precond is None else (lambda v: precond.apply(v, torch.empty_like(v)))  # noqa: E731
    V = torch.zeros(m + 1, n, dtype=b.dtype, device=b.device)
    H = np.zeros((m + 1, m))
    it, cycles, relres = 0, 0, 1.0
    while True:
        r = b - mv(x)
        beta = float(torch.linalg.vector_norm(r))
        syncs += 1
        relres = beta / bnorm
        if not np.isfinite(relres) or relres <= tol or it >= maxiter:
            break
        V[0] = r / beta
        g = np.zeros(m + 1)
        g[0] = beta
        cs, sn = np.zeros(m), np.zeros(m)
        k = 0
        for j in range(min(m, maxiter - it)):
            w = mv(prec(V[j]))
            h = torch.zeros(j + 1, dtype=b.dtype, device=b.device)
            for _ in range(2):                                     # CGS2
                hp = V[:j + 1] @ w
                w = w - V[:j + 1].T @ hp
                h = h + hp
            hv = torch.cat((h, torch.linalg.vector_norm(w).reshape(1))).cpu().numpy()     # one host read per step
            syncs += 1
            hn = float(hv[-1])
            col = np.zeros(m + 1)
            col[:j + 1] = hv[:-1]
            for i in range(j):
                col[i], col[i + 1] = cs[i] * col[i] + sn[i] * col[i + 1], -sn[i] * col[i] + cs[i] * col[i + 1]
            rr = float(np.hypot(col[j], hn))
            cs[j], sn[j] = (col[j] / rr, hn / rr) if rr > 0 else (1.0, 0.0)
            col[j], col[j + 1] = rr, 0.0
            g[j + 1], g[j] = -sn[j] * g[j], cs[j] * g[j]
            H[:, j] = col
            k = j + 1
            if not abs(g[j + 1]) > tol * bnorm or not hn > 1e-15 * rr:
                break
            V[j + 1] = w / hn
        it += k
        cycles += 1
        y = np.zeros(k)
        for i in range(k - 1, -1, -1):
            y[i] = (g[i] - H[i, i + 1:k] @ y[i + 1:k]) / H[i, i]
        x = x + prec(V[:k].T @ torch.as_tensor(y, dtype=b.dtype, device=b.device))
        if k == 0:
            break
    return x, {"iterations": it, "restarts": max(cycles - 1, 0), "relres": relres, "converged": bool(relres <= tol),
               "host_syncs": syncs}


def _gmres_fused(a, b, precond, x0, tol, restart, maxiter, check_every):
    """The GMRES loop on the device (csrc/gmres.cu): plain launches, no CUDA graph (the multi-column kernels change
    their width every step).  The host reads the scalar buffer once per ``check_every`` Arnoldi steps and once per
    restart (the true residual).  Once the DONE flag is set inside a block of steps, every GMRES kernel and the block
    apply of the remaining steps return at once; the SpMV (the shared ``pb_csr_spmv_dev``) does not read the flag, so
    up to ``check_every - 1`` SpMVs per solve run for nothing -- at most 7 against the 450-1800 steps of the measured
    contact problems."""
    import ctypes as C
    import torch
    from . import _lib
    lib = _lib.load()
    n = int(a.shape[0])
    if tuple(a.shape) != (n, n) or b.numel() != n:
        raise ValueError("gmres: a square matrix and a right-hand side of matching size are expected")
    if not b.is_cuda:
        raise RuntimeError("gmres: the device loop needs a CUDA right-hand side (no CPU path)")
    if precond is not None and precond.n != n:
        raise ValueError("gmres: the preconditioner's layout does not match the matrix")
    dev = b.device
    m = max(1, min(int(restart), n, 4096))
    check_every = max(1, int(check_every))
    b = b.contiguous().to(torch.float64)
    f64 = lambda k: torch.zeros(k, dtype=torch.float64, device=dev)  # noqa: E731
    x = f64(n) if x0 is None else x0.to(torch.float64).clone().contiguous()
    V = torch.zeros((m + 1) * n, dtype=torch.float64, device=dev)
    z, t = f64(n), f64(n)
    H, hb, cs, sn, g, y = f64((m + 1) * m), f64(2 * (m + 1) + 2), f64(m), f64(m), f64(m + 1), f64(m)
    scal = f64(8)
    done = C.c_void_p(scal.data_ptr() + 8 * 5)                     # the sticky DONE flag (GS_DONE in gmres.cu)
    P = lambda q: C.c_void_p(q.data_ptr())  # noqa: E731
    A = lambda off: C.c_void_p(V.data_ptr() + 8 * off)  # noqa: E731
    col = lambda j: A(j * n)  # noqa: E731
    st = torch.cuda.current_stream().cuda_stream
    ck = _lib.check
    syncs, it, cycles, relres, bnorm = 0, 0, 0, 1.0, None
    v0 = V[:n]
    while True:
        # true residual r = b - A x into V[:, 0]
        scal[1].zero_()
        a.spmv_device(x.data_ptr(), V.data_ptr(), st)
        ck(lib.pb_gm_residual(n, P(b), P(V), P(scal), int(bnorm is None), st))
        ck(lib.pb_gm_start(m, float(tol), P(hb), P(g), P(scal), st))
        h = scal.cpu().numpy()
        syncs += 1
        if bnorm is None:
            bnorm = float(np.sqrt(max(h[0], 0.0)))
            if bnorm == 0.0:
                x.zero_()
                return x, {"iterations": 0, "restarts": 0, "relres": 0.0, "converged": True, "host_syncs": syncs,
                           "cuda_graph": False}
        relres = float(np.sqrt(max(h[1], 0.0))) / bnorm
        if not np.isfinite(relres) or relres <= tol or it >= maxiter:
            break
        ck(lib.pb_gm_scale(n, P(v0), P(scal), st))
        steps = min(m, maxiter - it)
        k = 0
        for j in range(steps):
            if precond is not None:
                ck(lib.pb_local_block_apply_dev(*precond._args(), P(precond.inv), col(j), P(z), done, st))
                src = z.data_ptr()
            else:
                src = V.data_ptr() + 8 * j * n
            a.spmv_device(src, V.data_ptr() + 8 * (j + 1) * n, st)
            for p in range(2):
                hp = C.c_void_p(hb.data_ptr() + 8 * p * (m + 1))
                ww = C.c_void_p(hb.data_ptr() + 8 * (2 * (m + 1) + p))
                ck(lib.pb_gm_dots(n, P(V), j + 1, col(j + 1), hp, P(scal), st))
                ck(lib.pb_gm_orth(n, P(V), j + 1, hp, col(j + 1), ww, P(scal), st))
            ck(lib.pb_gm_givens(j, m, P(H), P(hb), P(cs), P(sn), P(g), P(scal), st))
            ck(lib.pb_gm_scale(n, col(j + 1), P(scal), st))
            if (j + 1) % check_every == 0 or j + 1 == steps:
                h = scal.cpu().numpy()
                syncs += 1
                k = int(h[6])
                if h[5] != 0.0:
                    break
        it += k
        cycles += 1
        ck(lib.pb_gm_ysolve(m, P(H), P(g), P(y), P(scal), st))
        if precond is not None:
            ck(lib.pb_gm_combine(n, P(V), m, P(y), P(t), P(scal), 0, st))
            ck(lib.pb_local_block_apply_dev(*precond._args(), P(precond.inv), P(t), P(z), None, st))
            ck(lib.pb_gm_axpy(n, P(z), P(x), st))
        else:
            ck(lib.pb_gm_combine(n, P(V), m, P(y), P(x), P(scal), 1, st))
        if k == 0:
            break
    return x, {"iterations": it, "restarts": max(cycles - 1, 0), "relres": relres, "converged": bool(relres <= tol),
               "host_syncs": syncs, "cuda_graph": False}
