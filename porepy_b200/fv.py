"""Finite-volume discretizations behind PorePy's ``Discretization`` operator API, executed
by the sm_100a kernels of libporeb200.so.

Mirrors (same constructor, attribute names, matrix-dictionary keys, parameter keys and
exceptions) of

* ``pp.Mpfa``   reference src/porepy/numerics/fv/mpfa.py:29  (``discretize`` :65) with the
  ``FVElliptic`` base (numerics/fv/fv_elliptic.py:16, ``assemble_matrix_rhs`` :67-112),
* ``pp.Mpsa``   reference src/porepy/numerics/fv/mpsa.py:38  (``discretize`` :121,
  ``assemble_matrix_rhs`` :486-529),
* ``pp.Biot``   reference src/porepy/numerics/fv/biot.py:40  (``discretize`` :247).

Inputs come from ``data["parameters"][keyword]``, outputs (scipy CSR) go to
``data["discretization_matrices"][keyword][<key>]`` exactly as in the reference, so the classes
drop into ``EquationSystem.discretize`` / the model mixins (see porepy_b200/porepy_plugin.py
for the ``pp.ad.MpfaAd`` subclasses used when the reference is importable).

There is no CPU path: without the built CUDA library or without a GPU every ``discretize``
raises ``RuntimeError``.
"""
from __future__ import annotations

import ctypes as C
import logging
import time

import numpy as np
import scipy.sparse as sps

from . import _lib
from .params import DISCRETIZATION_MATRICES, PARAMETERS

logger = logging.getLogger(__name__)


def determine_eta(sd) -> float:
    """numerics/fv/_fvutils.py:280-305: 1/3 on simplex grids, 0 otherwise."""
    name = getattr(sd, "name", "")
    if not isinstance(name, str):
        name = " ".join(str(n) for n in name)
    return 1.0 / 3.0 if ("TriangleGrid" in name or "TetrahedralGrid" in name) else 0.0


def block_expand(ip: np.ndarray, ix: np.ndarray, br: int, bc: int):
    """Expand a base pattern into br x bc blocks (row r*br+i, column c*bc+j).  The value of
    block entry (i, j) of base entry p in base row r is stored at
    ``br*bc*ip[r] + i*bc*len_r + (p-ip[r])*bc + j`` -- the layout the kernels scatter into."""
    ip = ip.astype(np.int64)
    lens = np.diff(ip)
    new_ip = np.zeros(lens.size * br + 1, dtype=np.int64)
    np.cumsum(np.repeat(lens * bc, br), out=new_ip[1:])
    cols = ix.astype(np.int64)
    if bc > 1:
        cols = (cols[:, None] * bc + np.arange(bc, dtype=np.int64)).reshape(-1)
    if br == 1:
        return new_ip, cols
    out = np.empty(new_ip[-1], dtype=np.int64)
    rep = lens * bc
    row_of = np.repeat(np.arange(lens.size, dtype=np.int64), rep)
    off = np.arange(cols.size, dtype=np.int64) - np.repeat(ip[:-1] * bc, rep)
    for i in range(br):
        out[new_ip[row_of * br + i] + off] = cols
    return new_ip, out


def _index_dtype(nnz: int, ncols: int):
    return np.int32 if max(nnz, ncols) < 2**31 - 1 else np.int64


# ------------------------------------------------------------------------------------------
# 2-D grids embedded in 3-D (fracture planes)
# ------------------------------------------------------------------------------------------


def plane_frame(sd, tol: float = 1e-5):
    """Rotation ``R`` (3, 3) with rows (t1, t2, n) that maps a planar 2-D grid into its own
    plane, or ``None`` when the grid already lies in a plane z = const.

    The reference rotates such grids with ``map_geometry.map_grid`` before discretizing
    (numerics/fv/mpfa.py:733-754).  Any in-plane basis gives the same matrices (the scheme is
    invariant under rotations and reflections), so the frame is taken from the principal axes
    of the node cloud."""
    x = np.asarray(sd.nodes, dtype=np.float64)
    xc = x - x.mean(axis=1, keepdims=True)
    w, v = np.linalg.eigh(xc @ xc.T)          # ascending: v[:, 0] is the plane normal
    n = v[:, 0]
    extent = np.sqrt(max(w[2], 0.0) / max(x.shape[1], 1)) + 1e-300
    if np.abs(n @ xc).max() > tol * max(extent, np.abs(xc).max()):
        raise ValueError("2-D grid is not planar")
    if abs(abs(n[2]) - 1.0) <= 1e-14 and np.ptp(x[2]) <= 1e-12 * max(1.0, np.abs(x).max()):
        return None
    t1 = v[:, 2]
    t2 = np.cross(n, t1)
    return np.vstack((t1, t2 / np.linalg.norm(t2), n))


def plan_geometry(sd):
    """The six geometry arrays the plan reads, and the rotation applied to them (None for 3-D
    grids and for 2-D grids in a plane z = const)."""
    arrs = [sd.nodes, sd.face_normals, sd.face_centers, sd.face_areas, sd.cell_centers, sd.cell_volumes]
    rot = plane_frame(sd) if int(sd.dim) == 2 else None
    if rot is not None:
        for i in (0, 1, 2, 4):
            a = rot @ np.asarray(arrs[i], dtype=np.float64)
            a[2] = 0.0
            arrs[i] = a
    return [_lib.f64(a) for a in arrs], rot


def rotate_second_order(values: np.ndarray, rot: np.ndarray) -> np.ndarray:
    """R K R^T per cell for (3, 3, nc) values (mpfa.py:749-754; the kernels read the leading
    nd x nd block)."""
    return np.einsum("ia,abc,jb->ijc", rot, np.asarray(values, dtype=np.float64), rot)


def lift_vector_source(ip: np.ndarray, ix: np.ndarray, data: np.ndarray, rows: np.ndarray, nc: int):
    """(nf, 2 nc) vector-source matrix in the plane's coordinates -> (nf, amb nc) in the ambient space
    (amb = ``rows.shape[1]``, 2 or 3): every (face, cell) pair of in-plane coefficients is multiplied by the
    two in-plane rows of the rotation, restricted to the first ``amb`` ambient components (mpfa.py:423-466).
    ``ip, ix`` is the FACE x CELL base pattern, ``data`` holds the two coefficients of each base entry
    consecutively."""
    rows = np.asarray(rows, dtype=np.float64)
    amb = rows.shape[1]
    da = np.asarray(data, dtype=np.float64).reshape(-1, 2) @ rows
    dt = _index_dtype(amb * int(ix.size), amb * nc)
    cols = (ix.astype(dt)[:, None] * amb + np.arange(amb, dtype=dt)).ravel()
    return sps.csr_matrix((da.ravel(), cols, ip.astype(dt) * amb), shape=(ip.size - 1, amb * nc))


def _log_throughput(name: str, keyword: str, sd, kernel_ms: float, wall_s: float, out: dict) -> None:
    """One INFO line per discretization (the reference logs the elapsed time of ``discretize``,
    models/solution_strategy.py:435-441): cells/s of the kernels and of the whole call, and the rate at which the
    output values were written."""
    if not logger.isEnabledFor(logging.INFO):
        return
    nbytes = 0
    for m in out.values():
        for mm in (m.values() if isinstance(m, dict) else (m,)):
            nbytes += 8 * int(getattr(mm, "nnz", 0))
    k_s = max(kernel_ms, 1e-6) * 1e-3
    logger.info("B200 %s(%s): %d cells (dim %d), kernels %.2f ms = %.3g cells/s, %.1f GB/s of output values; "
                "discretize() %.3f s = %.3g cells/s", name, keyword, sd.num_cells, sd.dim, kernel_ms,
                sd.num_cells / k_s, nbytes / k_s / 1e9, wall_s, sd.num_cells / max(wall_s, 1e-9))


def _on_device(*mats) -> bool:
    """All given matrices are ``LazyCsr`` whose values still live only on the device (untouched by the host)."""
    from .sparse import LazyCsr
    return all(isinstance(m, LazyCsr) and m.device_values is not None and not m.on_host for m in mats)


def _lazy_system(a_dev):
    """scipy-compatible view of a device-assembled system matrix; downloaded on first touch."""
    from .sparse import LazyCsr
    cache = {}

    def host():
        if "m" not in cache:
            cache["m"] = a_dev.to_scipy()
        return cache["m"]
    return LazyCsr.lazy(a_dev.shape, a_dev.nnz, lambda: host().data, lambda: host().indices, lambda: host().indptr,
                        device_csr=a_dev)


def _lifted(plan, m, rows: np.ndarray, nc: int):
    """``lift_vector_source`` of the (possibly still device-resident) in-plane matrix ``m``, itself lazy: the
    lifting runs on the host when the lifted matrix is first touched.  Keeps the in-plane device values and the
    rotation rows for ``assemble_matrix_rhs`` (which rotates the vector instead of the matrix)."""
    from .sparse import LazyCsr
    amb = rows.shape[1]
    cache = {}

    def built():
        if "m" not in cache:
            ip, ix = plan.base_pattern(0)
            cache["m"] = lift_vector_source(ip, ix, m.data, rows, nc)
        return cache["m"]
    out = LazyCsr.lazy((m.shape[0], amb * nc), (m.nnz // 2) * amb, lambda: built().data, lambda: built().indices,
                       lambda: built().indptr, device_values=getattr(m, "device_values", None), plan=plan)
    out.__dict__["plane_rows"] = rows
    return out


NUM_SOLVER_CFGS = 8


def solver_limits(cfg: int) -> tuple:
    """``(team, max_n, max_w)`` of dense solver configuration ``cfg`` (0..7): threads per system, the largest
    system order and the largest augmented width ``n + nrhs`` (2**31 - 1 for the catch-all configuration 6)."""
    lib = _lib.load()
    team, mn, mw = C.c_int(), C.c_int(), C.c_int()
    _lib.check(lib.pb_solver_limits(int(cfg), C.byref(team), C.byref(mn), C.byref(mw)))
    return team.value, mn.value, mw.value


def local_solve_batch(cfg: int, A, n: int, a_global: bool = False):
    """Solve the augmented systems ``A`` (shape (nsys, n, n + nrhs): ``[M | B]``) on the device with dense solver
    configuration ``cfg``, exactly as the assembly kernels run it on an interaction region.  Returns ``(X, ok)``:
    X (nsys, n, nrhs) = M^-1 B (NaN where the solver refused the system), ok (nsys,) bool."""
    lib = _lib.load()
    A = np.ascontiguousarray(A, dtype=np.float64)
    if A.ndim != 3 or A.shape[1] != n or A.shape[2] <= n:
        raise ValueError("A must have shape (nsys, n, n + nrhs) with nrhs >= 1")
    nsys, nrhs = A.shape[0], A.shape[2] - n
    X = np.empty((nsys, n, nrhs), np.float64)
    ok = np.empty(nsys, np.int32)
    _lib.check(lib.pb_local_solve_batch(int(cfg), int(bool(a_global)), nsys, int(n), int(nrhs),
                                        _lib.ptr(A, _lib._f64p), _lib.ptr(X, _lib._f64p), _lib.ptr(ok, _lib._i32p)))
    return X, ok.astype(bool)


class DevicePlan:
    """Device-resident sub-cell topology + output patterns of one grid (``pb_plan``).

    Built once per grid topology and cached on the grid object; MPFA, MPSA and Biot share it.
    """

    def __init__(self, sd):
        lib = _lib.load()
        _lib.require_gpu()
        self.lib = lib
        if hasattr(sd, "periodic_face_map"):
            raise NotImplementedError("periodic faces are not supported by porepy_b200")
        if sd.dim not in (2, 3):
            raise NotImplementedError(
                f"porepy_b200 discretizes 2-D and 3-D grids; dim={sd.dim} (TPFA fallback of "
                "mpfa.py:690-712) is not part of this build")
        cf = sps.csc_matrix(sd.cell_faces)
        fn = sps.csc_matrix(sd.face_nodes)
        self.nd, self.nc, self.nf, self.nn = int(sd.dim), sd.num_cells, sd.num_faces, sd.num_nodes
        i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)  # noqa: E731  (no copy when scipy already holds int32)
        cfp, cfi = i32(cf.indptr), i32(cf.indices)
        cfd = np.asarray(cf.data).astype(np.int8)
        fnp, fni = i32(fn.indptr), i32(fn.indices)
        h = C.c_void_p()
        t0 = time.perf_counter()
        _lib.check(lib.pb_plan_create(self.nd, self.nc, self.nf, self.nn,
                                      _lib.ptr(cfp, _lib._i32p), _lib.ptr(cfi, _lib._i32p),
                                      _lib.ptr(cfd, _lib._i8p), _lib.ptr(fnp, _lib._i32p),
                                      _lib.ptr(fni, _lib._i32p), C.byref(h)))
        self.plan_seconds = time.perf_counter() - t0
        self.h = h
        self.fingerprint = self._fingerprint(sd, cf, fn)
        self._base = {}
        self._expanded = {}
        self.rotation = None

    def __del__(self):
        h = getattr(self, "h", None)
        if h is not None and h.value:
            try:
                self.lib.pb_plan_destroy(h)
            except Exception:
                pass
            self.h = None

    @staticmethod
    def _fingerprint(sd, cf, fn):
        """Counts plus a strided checksum of the index arrays: a topology edit that keeps the counts (split faces
        renumbered, ...) must not reuse a stale plan."""
        ci, fi = np.asarray(cf.indices), np.asarray(fn.indices)
        return (int(sd.dim), sd.num_cells, sd.num_faces, sd.num_nodes, int(cf.nnz), int(fn.nnz),
                int(ci[::7].astype(np.int64).sum()), int(fi[::7].astype(np.int64).sum()),
                int(np.asarray(cf.indptr)[::5].astype(np.int64).sum()))

    @classmethod
    def for_grid(cls, sd) -> "DevicePlan":
        cf, fn = sd.cell_faces, sd.face_nodes
        fp = cls._fingerprint(sd, cf, fn)
        plan = getattr(sd, "_b200_plan", None)
        if plan is None or plan.fingerprint != fp:
            plan = cls(sd)
            try:
                sd._b200_plan = plan
            except AttributeError:
                pass
        plan.set_geometry(sd)
        return plan

    def set_geometry(self, sd) -> None:
        """Upload the geometry.  2-D grids embedded in 3-D are rotated into their own plane first
        (``plan_geometry``); ``self.rotation`` keeps the rotation for the callers."""
        arrs, self.rotation = plan_geometry(sd)
        _lib.check(self.lib.pb_plan_set_geometry(self.h, *[_lib.ptr(a, _lib._f64p) for a in arrs]))

    def set_cell_map(self, cells, n_source_cells: int) -> None:
        """Cell ``e`` of this plan is cell ``cells[e]`` of a larger grid with ``n_source_cells`` cells: the cell
        tensors of the following uploads may then be the arrays of THAT grid (shape (3, 3, n_source) / (9, 9,
        n_source)); they are restricted on the device.  A shard passes the global tensors as they are."""
        if cells is None:
            _lib.check(self.lib.pb_plan_set_cell_map(self.h, None, 0))
            self.n_source_cells = None
            return
        m = np.ascontiguousarray(cells, dtype=np.int64)
        if m.shape != (self.nc,):
            raise ValueError("cell map must have one entry per cell of this plan")
        _lib.check(self.lib.pb_plan_set_cell_map(self.h, _lib.ptr(m, _lib._i64p), int(n_source_cells)))
        self.n_source_cells = int(n_source_cells)
        self._cell_map_host = m

    def _cells_of(self, arr) -> bool:
        """True when a cell tensor has the source grid's size and must go through the cell map (clears the map when
        the caller passes arrays of this plan's own size instead)."""
        n = arr.shape[-1]
        src = getattr(self, "n_source_cells", None)
        if src is not None and n == src and n != self.nc:
            return True
        if src is not None and n == self.nc:
            self.set_cell_map(None, 0)
        return False

    def set_active_nodes(self, mask) -> None:
        """Assemble only the interaction regions of the flagged nodes (``None``: all).  The multi-GPU path flags
        a shard's own nodes: the outer nodes of its halo layer are incomplete and their rows are discarded."""
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        if m is not None and m.shape != (self.nn,):
            raise ValueError("active-node mask must have one entry per node")
        _lib.check(self.lib.pb_plan_set_active_nodes(self.h, _lib.ptr(m, _lib._u8p)))

    # ---- patterns
    def base_pattern(self, which: int):
        if which not in self._base:
            nr, nz = C.c_int64(), C.c_int64()
            _lib.check(self.lib.pb_plan_pattern_size(self.h, which, C.byref(nr), C.byref(nz)))
            ip = np.zeros(nr.value + 1, np.int32)
            ix = np.zeros(max(nz.value, 1), np.int32)
            _lib.check(self.lib.pb_plan_pattern_get(self.h, which, _lib.ptr(ip, _lib._i32p),
                                                    _lib.ptr(ix, _lib._i32p)))
            ix = ix[:nz.value]
            ip.flags.writeable = ix.flags.writeable = False   # shared by every matrix on this grid
            self._base[which] = (ip, ix)
        return self._base[which]

    def nnz(self, which: int) -> int:
        return int(self.base_pattern(which)[1].size)

    def pattern(self, which: int, br: int, bc: int):
        key = (which, br, bc)
        if key not in self._expanded:
            ip, ix = self.base_pattern(which)
            if br == 1 and bc == 1:
                self._expanded[key] = (ip, ix)
            else:
                ncols = {0: self.nc, 1: self.nf, 2: self.nc, 3: self.nf}[which] * bc
                nnz = int(ix.size) * br * bc
                if max(nnz, ncols) < 2**31 - 1:
                    # expansion on the device, D2H into page-locked buffers
                    nip = _lib.pinned_empty((ip.size - 1) * br + 1, np.int32)
                    nix = _lib.pinned_empty(max(nnz, 1), np.int32)
                    _lib.check(self.lib.pb_plan_pattern_expanded(
                        self.h, which, br, bc, _lib.ptr(nip, _lib._i32p), _lib.ptr(nix, _lib._i32p)))
                    nix = nix[:nnz]
                else:  # beyond int32: host expansion with 64-bit indices
                    nip, nix = block_expand(ip, ix, br, bc)
                nip.flags.writeable = nix.flags.writeable = False
                self._expanded[key] = (nip, nix)
        return self._expanded[key]

    def matrix(self, which: int, br: int, bc: int, data: np.ndarray) -> sps.csr_matrix:
        ip, ix = self.pattern(which, br, bc)
        nrows = (ip.size - 1)
        ncols = {0: self.nc, 1: self.nf, 2: self.nc, 3: self.nf}[which] * bc
        m = sps.csr_matrix((data, ix, ip), shape=(nrows, ncols), copy=False)
        m.has_sorted_indices = True
        return m

    def sizes(self) -> dict:
        a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
        d, e = C.c_int32(), C.c_int32()
        _lib.check(self.lib.pb_plan_sizes(self.h, C.byref(a), C.byref(b), C.byref(c), C.byref(d),
                                          C.byref(e)))
        return dict(subcells=a.value, subfaces=b.value, subhalffaces=c.value,
                    max_subfaces_per_node=d.value, max_subcells_per_node=e.value)

    def node_classes(self, kind: str) -> list:
        """The node classes of the last build for ``kind`` ("mpfa", or "mpsa" for MPSA and Biot): a list of
        ``(cfg, a_global, num_nodes)``, one per class, where ``cfg`` is the dense solver configuration its nodes
        run (see ``solver_limits``) and ``a_global`` whether their matrices live in global memory."""
        k = {"mpfa": 0, "mpsa": 1}[kind]
        n = C.c_int()
        _lib.check(self.lib.pb_plan_node_classes(self.h, k, 0, None, None, None, C.byref(n)))
        cfg = np.zeros(max(n.value, 1), np.int32)
        glob = np.zeros(max(n.value, 1), np.uint8)
        nodes = np.zeros(max(n.value, 1), np.int64)
        _lib.check(self.lib.pb_plan_node_classes(self.h, k, n.value, _lib.ptr(cfg, _lib._i32p),
                                                 _lib.ptr(glob, _lib._u8p), _lib.ptr(nodes, _lib._i64p),
                                                 C.byref(n)))
        return [(int(cfg[i]), bool(glob[i]), int(nodes[i])) for i in range(n.value)]

    # ---- MPFA
    def mpfa_upload(self, perm, codes, robw, eta) -> None:
        perm = _lib.f64(perm)
        if not self._cells_of(perm) and perm.shape != (3, 3, self.nc):
            raise ValueError("second_order_tensor.values must have shape (3, 3, num_cells)")
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        robw = None if robw is None else _lib.f64(robw)
        _lib.check(self.lib.pb_mpfa_upload(self.h, _lib.ptr(perm, _lib._f64p),
                                           _lib.ptr(codes, _lib._u8p), _lib.ptr(robw, _lib._f64p),
                                           float(eta)))

    def mpfa_assemble(self, flux=True, trace=True, vector_source=True) -> float:
        ms = C.c_float()
        _lib.check(self.lib.pb_mpfa_assemble(self.h, int(flux), int(trace), int(vector_source),
                                             C.byref(ms)))
        return float(ms.value)

    def mpfa_download(self, flux=True, trace=True, vector_source=True) -> dict:
        nd = self.nd
        nfc, nfb = self.nnz(0), self.nnz(1)
        bufs = {
            "flux": _lib.pinned_empty(nfc) if flux else None,
            "bound_flux": _lib.pinned_empty(nfb) if flux else None,
            "bound_pressure_cell": _lib.pinned_empty(nfc) if trace else None,
            "bound_pressure_face": _lib.pinned_empty(nfb) if trace else None,
            "vector_source": _lib.pinned_empty(nfc * nd) if (flux and vector_source) else None,
            "bound_pressure_vector_source": _lib.pinned_empty(nfc * nd) if (trace and vector_source) else None,
        }
        _lib.check(self.lib.pb_mpfa_download(self.h, *[_lib.ptr(b, _lib._f64p) for b in bufs.values()]))
        shape = {"flux": (0, 1, 1), "bound_flux": (1, 1, 1), "bound_pressure_cell": (0, 1, 1),
                 "bound_pressure_face": (1, 1, 1), "vector_source": (0, 1, nd),
                 "bound_pressure_vector_source": (0, 1, nd)}
        return {k: self.matrix(*shape[k], v) for k, v in bufs.items() if v is not None}

    # ---- device-resident results (lazily downloaded scipy matrices)
    def _ncols(self, which: int, bc: int) -> int:
        return {0: self.nc, 1: self.nf, 2: self.nc, 3: self.nf}[which] * bc

    def take(self, key: int):
        """Move the value array of output ``key`` (``PB_OUT_*``) out of the plan; it stays in HBM."""
        from .sparse import DeviceValues
        h = C.c_void_p()
        _lib.check(self.lib.pb_plan_take_output(self.h, int(key), C.byref(h)))
        return DeviceValues(h, self.lib)

    def lazy_matrix(self, key: int, which: int, br: int, bc: int):
        """Output ``key`` as a ``LazyCsr`` on pattern ``which`` expanded to br x bc blocks: values, indices and
        row pointers are downloaded when (and if) a caller touches them."""
        from .sparse import LazyCsr
        vals = self.take(key)
        nrows = {0: self.nf, 1: self.nf, 2: self.nc, 3: self.nc}[which] * br
        pat_nnz = {w: None for w in range(4)}
        nr, nz = C.c_int64(), C.c_int64()
        _lib.check(self.lib.pb_plan_pattern_size(self.h, which, C.byref(nr), C.byref(nz)))
        del pat_nnz
        m = LazyCsr.lazy((nrows, self._ncols(which, bc)), nz.value * br * bc, vals.download,
                         lambda: self.pattern(which, br, bc)[1], lambda: self.pattern(which, br, bc)[0],
                         device_values=vals, plan=self)
        m.__dict__["pattern_key"] = (which, br, bc)
        return m

    def output_csr(self, values, which: int, br: int, bc: int):
        """A detached output as a ``DeviceCsr`` (block-expanded pattern + a copy of the values), the operand form of
        the device-side AD chain (``porepy_b200.ad``)."""
        from .sparse import DeviceCsr
        h = C.c_void_p()
        _lib.check(self.lib.pb_plan_output_csr(self.h, values.h, which, br, bc, C.byref(h)))
        return DeviceCsr.from_handle(h)

    def mpfa_lazy(self, flux=True, trace=True, vector_source=True) -> dict:
        nd = self.nd
        spec = {"flux": (0, 0, 1, flux), "bound_flux": (1, 1, 1, flux), "bound_pressure_cell": (2, 0, 1, trace),
                "bound_pressure_face": (3, 1, 1, trace), "vector_source": (4, 0, nd, flux and vector_source),
                "bound_pressure_vector_source": (5, 0, nd, trace and vector_source)}
        return {k: self.lazy_matrix(key, which, 1, bc) for k, (key, which, bc, want) in spec.items() if want}

    def mpsa_lazy(self) -> dict:
        nd = self.nd
        return {"stress": self.lazy_matrix(6, 0, nd, nd), "bound_stress": self.lazy_matrix(7, 1, nd, nd),
                "bound_displacement_cell": self.lazy_matrix(8, 0, nd, nd),
                "bound_displacement_face": self.lazy_matrix(9, 1, nd, nd)}

    def biot_lazy(self, q: int) -> dict:
        nd, b = self.nd, 10 + 5 * q
        return {"displacement_divergence": self.lazy_matrix(b, 2, 1, nd),
                "boundary_displacement_divergence": self.lazy_matrix(b + 1, 3, 1, nd),
                "scalar_gradient": self.lazy_matrix(b + 2, 0, nd, 1),
                "mpsa_consistency": self.lazy_matrix(b + 3, 2, 1, 1),
                "bound_displacement_pressure": self.lazy_matrix(b + 4, 0, nd, 1)}

    @staticmethod
    def _vh(values):
        return None if values is None else values.h

    def mpfa_system(self, flux=None):
        """A = div @ flux assembled and kept on the device (``DeviceCsr``) from the flux values given as a
        ``DeviceValues`` handle (``None``: the plan's last assembled array)."""
        from .sparse import DeviceCsr
        h = C.c_void_p()
        _lib.check(self.lib.pb_mpfa_system(self.h, self._vh(flux), C.byref(h)))
        return DeviceCsr.from_handle(h)

    def mpfa_rhs(self, bc_values, vector_source=None, bound_flux=None, vector_source_discr=None) -> np.ndarray:
        """b = -div @ (bound_flux @ bc_values) [- div @ (vector_source_discr @ vector_source)]."""
        bv = _lib.f64(bc_values)
        vs = None if vector_source is None else _lib.f64(vector_source)
        rhs = np.empty(self.nc)
        _lib.check(self.lib.pb_mpfa_rhs(self.h, self._vh(bound_flux), self._vh(vector_source_discr),
                                        _lib.ptr(bv, _lib._f64p), _lib.ptr(vs, _lib._f64p),
                                        _lib.ptr(rhs, _lib._f64p)))
        return rhs

    def mpsa_system(self, stress=None):
        """A = div_nd @ stress assembled and kept on the device (``DeviceCsr``)."""
        from .sparse import DeviceCsr
        h = C.c_void_p()
        _lib.check(self.lib.pb_mpsa_system(self.h, self._vh(stress), C.byref(h)))
        return DeviceCsr.from_handle(h)

    def mpsa_rhs(self, bc_values, source=None, bound_stress=None) -> np.ndarray:
        """b = -div_nd @ (bound_stress @ bc_values) + source   (mpsa.py:486-529)."""
        bv = _lib.f64(bc_values)
        src = None if source is None else _lib.f64(source)
        rhs = np.empty(self.nc * self.nd)
        _lib.check(self.lib.pb_mpsa_rhs(self.h, self._vh(bound_stress), _lib.ptr(bv, _lib._f64p),
                                        _lib.ptr(src, _lib._f64p), _lib.ptr(rhs, _lib._f64p)))
        return rhs

    # ---- MPSA / Biot
    def mpsa_upload(self, stiff, codes, robw, eta, alphas=()) -> None:
        stiff = _lib.f64(stiff)
        mapped = self._cells_of(stiff)
        if not mapped and stiff.shape != (9, 9, self.nc):
            raise ValueError("fourth_order_tensor.values must have shape (9, 9, num_cells)")
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        robw = None if robw is None else _lib.f64(robw)
        nal = len(alphas)
        al = None
        if nal:
            al = np.zeros((nal, 3, 3, self.n_source_cells if mapped else self.nc))
            for q, a in enumerate(alphas):
                a = np.asarray(a)
                if mapped and a.shape[-1] == self.nc:      # a tensor given for this plan's own cells
                    al[q][..., self._cell_map_host] = a
                else:
                    al[q] = a
        _lib.check(self.lib.pb_mpsa_upload(self.h, _lib.ptr(stiff, _lib._f64p),
                                           _lib.ptr(codes, _lib._u8p), _lib.ptr(robw, _lib._f64p),
                                           float(eta), nal, _lib.ptr(al, _lib._f64p)))
        self._nal = nal

    def mpsa_set_basis(self, basis) -> None:
        """``bc.basis`` (nd, nd, nf) or None for the identity; call after ``mpsa_upload``."""
        b = None if basis is None else _lib.f64(basis)
        if b is not None and b.shape != (self.nd, self.nd, self.nf):
            raise ValueError("bc.basis must have shape (nd, nd, num_faces)")
        _lib.check(self.lib.pb_mpsa_set_basis(self.h, _lib.ptr(b, _lib._f64p)))

    def mpsa_assemble(self) -> float:
        ms = C.c_float()
        _lib.check(self.lib.pb_mpsa_assemble(self.h, C.byref(ms)))
        return float(ms.value)

    def mpsa_download(self) -> dict:
        nd = self.nd
        nd2 = nd * nd
        nfc, nfb = self.nnz(0), self.nnz(1)
        bufs = [_lib.pinned_empty(nfc * nd2), _lib.pinned_empty(nfb * nd2), _lib.pinned_empty(nfc * nd2),
                _lib.pinned_empty(nfb * nd2)]
        _lib.check(self.lib.pb_mpsa_download(self.h, *[_lib.ptr(b, _lib._f64p) for b in bufs]))
        return {
            "stress": self.matrix(0, nd, nd, bufs[0]),
            "bound_stress": self.matrix(1, nd, nd, bufs[1]),
            "bound_displacement_cell": self.matrix(0, nd, nd, bufs[2]),
            "bound_displacement_face": self.matrix(1, nd, nd, bufs[3]),
        }

    def biot_download(self, q: int) -> dict:
        nd = self.nd
        nfc, ncc, ncb = self.nnz(0), self.nnz(2), self.nnz(3)
        bufs = [_lib.pinned_empty(ncc * nd), _lib.pinned_empty(ncb * nd), _lib.pinned_empty(nfc * nd),
                _lib.pinned_empty(ncc), _lib.pinned_empty(nfc * nd)]
        _lib.check(self.lib.pb_biot_download(self.h, q, *[_lib.ptr(b, _lib._f64p) for b in bufs]))
        return {
            "displacement_divergence": self.matrix(2, 1, nd, bufs[0]),
            "boundary_displacement_divergence": self.matrix(3, 1, nd, bufs[1]),
            "scalar_gradient": self.matrix(0, nd, 1, bufs[2]),
            "mpsa_consistency": self.matrix(2, 1, 1, bufs[3]),
            "bound_displacement_pressure": self.matrix(0, nd, 1, bufs[4]),
        }


class FaceGrid:
    """Face-indexed device view of a grid of any dimension (``pb_facegrid``): the face -> cell table and
    the face normals / centres and cell centres -- all the per-face schemes (TPFA, upwinding) read.  No
    interaction-region plan is built, so 1-D grids (the reference's TPFA delegation, mpfa.py:690-712,
    mpsa.py:666-697) and 2-D grids anywhere in space work as they are."""

    def __init__(self, sd):
        lib = _lib.load()
        _lib.require_gpu()
        self.lib = lib
        if getattr(sd, "periodic_face_map", None) is not None:
            raise NotImplementedError("periodic faces are not supported by porepy_b200")
        cf = sps.csc_matrix(sd.cell_faces)
        self.nc, self.nf = sd.num_cells, sd.num_faces
        cfp, cfi = cf.indptr.astype(np.int32), cf.indices.astype(np.int32)
        cfd = np.asarray(cf.data).astype(np.int8)
        geo = [_lib.f64(a) for a in (sd.face_normals, sd.face_centers, sd.cell_centers)]
        h = C.c_void_p()
        _lib.check(lib.pb_facegrid_create(self.nc, self.nf, _lib.ptr(cfp, _lib._i32p), _lib.ptr(cfi, _lib._i32p),
                                          _lib.ptr(cfd, _lib._i8p), *[_lib.ptr(a, _lib._f64p) for a in geo],
                                          C.byref(h)))
        self.h = h

    @classmethod
    def for_grid(cls, sd) -> "FaceGrid":
        return cls(sd)

    def __del__(self):
        h = getattr(self, "h", None)
        if h is not None and h.value:
            try:
                self.lib.pb_facegrid_destroy(h)
            except Exception:
                pass
            self.h = None

    def tpfa(self, perm, bc_bits, fc_indptr, vdim: int) -> list:
        """Value arrays of the six TPFA terms in the pattern of ``cell_faces`` (CSR by face):
        [flux, bound_pressure_cell, vector_source, bound_pressure_vector_source] and the diagonals
        [bound_flux, bound_pressure_face]."""
        perm = _lib.f64(perm)
        if perm.shape != (3, 3, self.nc):
            raise ValueError("second_order_tensor.values must have shape (3, 3, num_cells)")
        bits = np.ascontiguousarray(bc_bits, dtype=np.uint8)
        ip = np.ascontiguousarray(fc_indptr, dtype=np.int32)
        nnz = int(ip[-1])
        out = [np.empty(nnz), np.empty(nnz), np.empty(nnz * vdim), np.empty(nnz * vdim), np.empty(self.nf),
               np.empty(self.nf)]
        _lib.check(self.lib.pb_tpfa(self.h, _lib.ptr(perm, _lib._f64p), _lib.ptr(bits, _lib._u8p),
                                    _lib.ptr(ip, _lib._i32p), int(vdim), *[_lib.ptr(a, _lib._f64p) for a in out]))
        return out

    def tpfa_diff(self, k_c, fc_indptr):
        """Differentiable TPFA (``pb_tpfa_diff``): half-face transmissibilities, face transmissibilities and
        dT_f/dk_c (9 values per half-face) for the cell-major 9 * nc permeability vector ``k_c``."""
        k = np.ascontiguousarray(k_c, dtype=np.float64).reshape(-1)
        ip = np.ascontiguousarray(fc_indptr, dtype=np.int32)
        nhf = int(ip[-1])
        t_hf, T, dT = np.empty(nhf), np.empty(self.nf), np.empty(nhf * 9)
        _lib.check(self.lib.pb_tpfa_diff(self.h, _lib.ptr(k, _lib._f64p), _lib.ptr(ip, _lib._i32p),
                                         _lib.ptr(t_hf, _lib._f64p), _lib.ptr(T, _lib._f64p), _lib.ptr(dT, _lib._f64p)))
        return t_hf, T, dT

    def upwind(self, darcy_flux, bc_bits):
        """Upstream cell per face (-1: face not in the matrix) and the two boundary diagonals."""
        q = _lib.f64(darcy_flux)
        bits = np.ascontiguousarray(bc_bits, dtype=np.uint8)
        up = np.empty(self.nf, np.int32)
        neu, dr = np.empty(self.nf), np.empty(self.nf)
        _lib.check(self.lib.pb_upwind(self.h, _lib.ptr(q, _lib._f64p), _lib.ptr(bits, _lib._u8p),
                                      _lib.ptr(up, _lib._i32p), _lib.ptr(neu, _lib._f64p), _lib.ptr(dr, _lib._f64p)))
        return up, neu, dr



# ------------------------------------------------------------------------------------------
# boundary-condition encoding
# ------------------------------------------------------------------------------------------


def scalar_bc_codes(bc, nf: int) -> np.ndarray:
    """Face codes for MPFA.  Internal (fracture) faces are Neumann (mpfa.py:1452-1454)."""
    internal = np.asarray(getattr(bc, "is_internal", np.zeros(nf, bool)), bool)
    codes = np.zeros(nf, np.uint8)
    codes[np.asarray(bc.is_neu, bool) | internal] = _lib.BC_NEU
    codes[np.asarray(bc.is_dir, bool) & ~internal] = _lib.BC_DIR
    codes[np.asarray(bc.is_rob, bool) & ~internal] = _lib.BC_ROB
    return codes


def face_bc_bits(bc, nf: int) -> np.ndarray:
    """Boundary byte of the per-face kernels (csrc/face_kernels.cuh): effective code in bits 0-1
    (internal faces count as Neumann, tpfa.py:187-188), the raw ``is_dir`` / ``is_neu`` flags in
    bits 2 / 3 (used as such by tpfa.py:221-225 and upwind.py:260-270)."""
    internal = np.asarray(getattr(bc, "is_internal", np.zeros(nf, bool)), bool)
    is_dir, is_neu, is_rob = (np.asarray(getattr(bc, k), bool) for k in ("is_dir", "is_neu", "is_rob"))
    bits = np.zeros(nf, np.uint8)
    bits[is_rob & ~internal] = _lib.BC_ROB
    bits[is_dir & ~internal] = _lib.BC_DIR
    bits[is_neu | internal] = _lib.BC_NEU
    bits |= (is_dir.astype(np.uint8) << 2) | (is_neu.astype(np.uint8) << 3)
    return bits


def vector_bc_codes(bc, nd: int, nf: int):
    if getattr(bc, "bc_type", "vectorial") != "vectorial":
        raise AttributeError("MPSA must be given a vectorial boundary condition")  # mpsa.py:823
    codes = np.zeros((nd, nf), np.uint8)
    codes[np.asarray(bc.is_neu, bool)[:nd]] = _lib.BC_NEU
    codes[np.asarray(bc.is_dir, bool)[:nd]] = _lib.BC_DIR
    codes[np.asarray(bc.is_rob, bool)[:nd]] = _lib.BC_ROB
    robw = None
    if np.any(codes == _lib.BC_ROB):
        rw = np.asarray(bc.robin_weight, float)
        robw = np.ascontiguousarray(rw[:nd, :nd])
    return codes, robw


def vector_bc_basis(bc, nd: int, codes=None):
    """``bc.basis`` (nd, nd, nf) when it is not the identity on some boundary face, else None
    (_fvutils.py:765-945: boundary conditions given in a rotated coordinate system).  The basis acts on the equations
    of boundary sub-faces only, so with the (nd, nf) condition ``codes`` of ``vector_bc_codes`` the test reads the
    flagged faces instead of all of the (nd, nd, nf) array (40 ms at 2 * 10^6 faces, in front of every MPSA call)."""
    basis = getattr(bc, "basis", None)
    if basis is None:
        return None
    b = np.asarray(basis, float)
    if b.ndim != 3:
        return None
    sub = b[:nd, :nd]
    eye = np.eye(nd)[:, :, None]
    if sub.strides[-1] == 0:        # one matrix broadcast over the faces (e.g. a restricted shard condition)
        if np.array_equal(sub[:, :, :1], eye):
            return None
    else:
        probe = sub if codes is None else sub[:, :, np.flatnonzero(np.asarray(codes).any(axis=0))]
        if np.array_equal(probe, np.broadcast_to(eye, probe.shape)):
            return None   # the identity on every (boundary) face: exact test; anything else IS a rotated basis
    return np.ascontiguousarray(b[:nd, :nd])


# ------------------------------------------------------------------------------------------
# discretization classes
# ------------------------------------------------------------------------------------------


def active_indices(sd, params: dict):
    """Cells of the sub-grid to discretize and faces whose rows are (re)computed, from
    ``specified_cells / specified_faces / specified_nodes`` (``_fvutils.find_active_indices``,
    _fvutils.py:308-355, and ``cell_ind_for_partial_update``, :1260-1462).  Cells mode: the faces
    touching a node of the given cells, and every cell touching a node of those faces.  Faces mode
    (split faces): the faces sharing a node with the given ones, and two layers of cells around
    them.  Nodes mode (gradual build-up): the cells touching the given nodes, and the faces all of
    whose nodes are given.  Writes ``active_cells`` / ``active_faces`` into ``params``."""
    nc, nf, nn = sd.num_cells, sd.num_faces, sd.num_nodes
    spec = [params.get(k) for k in ("specified_cells", "specified_faces", "specified_nodes")]
    if all(v is None for v in spec):
        cells, faces = np.arange(nc), np.arange(nf)
        params["active_cells"], params["active_faces"] = cells, faces
        return cells, faces
    fn = abs(sps.csr_matrix(sd.face_nodes)).astype(np.float64)      # nn x nf
    cf = abs(sps.csr_matrix(sd.cell_faces)).astype(np.float64)      # nf x nc
    cn = (fn @ cf).tocsr()                                          # nn x nc

    def mask(n, idx):
        m = np.zeros(n)
        m[np.asarray(idx, dtype=np.int64)] = 1.0
        return m

    active_faces = np.zeros(nf, bool)
    cell_ind = np.zeros(nc, bool)
    if spec[0] is not None:
        vert = (cn @ mask(nc, spec[0])) > 0
        active_faces |= (fn.T @ vert.astype(np.float64)) > 0
        vert |= (fn @ active_faces.astype(np.float64)) > 0
        cell_ind |= (cn.T @ vert.astype(np.float64)) > 0
    if spec[1] is not None:
        pvert = (fn @ mask(nf, spec[1])) > 0
        active_faces |= (fn.T @ pvert.astype(np.float64)) > 0
        anodes = (fn @ active_faces.astype(np.float64)) > 0
        pcells = (cn.T @ anodes.astype(np.float64)) > 0
        anodes |= (cn @ pcells.astype(np.float64)) > 0
        cell_ind |= (cn.T @ anodes.astype(np.float64)) > 0
    if spec[2] is not None:
        vert = mask(nn, spec[2])
        cell_ind |= (cn.T @ vert) > 0
        active_faces |= np.asarray(fn.T @ vert).ravel() == np.asarray(fn.sum(axis=0)).ravel()
    cells, faces = np.flatnonzero(cell_ind), np.flatnonzero(active_faces)
    params["active_cells"], params["active_faces"] = cells, faces
    return cells, faces


def _replace_rows(old, new, keep_entity: np.ndarray):
    """``old`` with the rows of the flagged entities (block rows) replaced by those of ``new``."""
    old = sps.csr_matrix(old)
    new = sps.csr_matrix(new)
    br = new.shape[0] // keep_entity.size
    stay = sps.diags(np.repeat(~keep_entity, br).astype(np.float64))
    return (stay @ old + new).tocsr()


class _Base:
    """numerics/discretization.py:12-121."""

    def __init__(self, keyword: str) -> None:
        self.keyword = keyword
        self.last_timing: dict = {}

    def __repr__(self) -> str:
        """numerics/discretization.py:21-25."""
        return f"Discretization of type {self.__class__.__name__} with keyword {self.keyword}"

    def _key(self) -> str:
        return self.keyword + "_"

    def discretize(self, sd, data: dict) -> None:
        """Full discretization, or -- with ``specified_cells / specified_faces / specified_nodes`` in
        the parameters -- the reference's partial one (mpfa.py:176-201,468-508; biot.py:326-342,
        614-712): the sub-grid of the active cells is discretized as a whole (same kernels), the rows
        of the active faces (and, for Biot's cell-row terms, of the cells next to them) are embedded
        in global numbering, all other rows are zero -- or, with ``update_discretization = True``,
        keep the values already stored.  ``active_cells`` / ``active_faces`` are written back to the
        parameter dictionary as the reference does (_fvutils.py:346-353)."""
        params = data[PARAMETERS][self.keyword]
        mats = data.setdefault(DISCRETIZATION_MATRICES, {}).setdefault(self.keyword, {})
        cells, faces = active_indices(sd, params)
        if cells.size == sd.num_cells and faces.size == sd.num_faces:
            mats.update(self._discretize_grid(sd, params))
            return
        from . import shard as _shard
        update = bool(params.get("update_discretization", False))
        keep_faces = np.zeros(sd.num_faces, bool)
        keep_faces[faces] = True
        if update:
            # Cell-row terms (Biot) sum over ALL nodes of a cell, and every cell sharing a node with a
            # modified one changes.  The reference replaces the rows of the cells next to an active face
            # although some of their nodes have cut interaction regions in its sub-grid (biot.py:627-632;
            # "update is not fully tested", biot.py:318-324).  Replacing stored rows must not corrupt
            # them: grow the sub-grid by one ring and replace exactly the rows of the cells all of whose
            # interaction regions are complete in it.
            cn = (abs(sps.csr_matrix(sd.face_nodes)) @ abs(sps.csr_matrix(sd.cell_faces))).tocsr()
            cn.data[:] = 1.0
            inside = np.zeros(sd.num_cells)
            inside[cells] = 1.0
            grown = (cn.T @ ((cn @ inside) > 0).astype(np.float64)) > 0
            complete_node = (cn @ grown.astype(np.float64)) == np.asarray(cn.sum(axis=1)).ravel()
            keep_cells = grown & ((cn.T @ (~complete_node).astype(np.float64)) == 0)
            cells = np.flatnonzero(grown)
        else:
            keep_cells = np.asarray(abs(sps.csr_matrix(sd.cell_faces)).T @ keep_faces.astype(np.float64)).ravel() > 0
        sub = _shard.extract_cells(sd, cells, keep_faces, keep_cells)
        local = _shard.restrict_parameters(params, sub)
        local.setdefault(self._eta_key, determine_eta(sd))
        out = {key: _shard.embed(sub, key, m) for key, m in self._discretize_grid(sub.grid, local).items()}
        if update:
            for key, new in out.items():
                keep = keep_faces if _shard._LAYOUT[key][0] == "face" else keep_cells
                if isinstance(new, dict):
                    mats[key] = {k: _replace_rows(mats[key][k], v, keep) for k, v in new.items()}
                else:
                    mats[key] = _replace_rows(mats[key], new, keep)
        else:
            mats.update(out)

    def update_discretization(self, sd, data: dict) -> None:
        """numerics/discretization.py:54: re-discretize (the partial path of ``discretize`` applies when
        ``specified_cells/faces/nodes`` are set)."""
        self.discretize(sd, data)

    def _check_unsupported(self, params: dict, sd=None) -> None:
        """``partition_arguments`` bound the reference's working set (``_fvutils.py:358-411``); the
        kernels stream over nodes and never materialise the global block-diagonal inverse, so the
        key is accepted and ignored.  Periodic face pairs
        (``_fvutils.py:95-140``) are not merged by the topology plan: refuse rather than discretize
        the pair as two boundaries."""
        if sd is not None and getattr(sd, "periodic_face_map", None) is not None:
            raise NotImplementedError("periodic boundaries (sd.periodic_face_map) are not supported")
        return None


class Mpfa(_Base):
    """MPFA-O flux discretization; see module docstring.  Matrix keys as fv_elliptic.py:29-53."""

    def __init__(self, keyword: str) -> None:
        super().__init__(keyword)
        self.flux_matrix_key = "flux"
        self.bound_flux_matrix_key = "bound_flux"
        self.bound_pressure_cell_matrix_key = "bound_pressure_cell"
        self.bound_pressure_face_matrix_key = "bound_pressure_face"
        self.vector_source_matrix_key = "vector_source"
        self.bound_pressure_vector_source_matrix_key = "bound_pressure_vector_source"

    def ndof(self, sd) -> int:
        return sd.num_cells

    _eta_key = "mpfa_eta"

    def _discretize_grid(self, sd, params: dict) -> dict:
        """mpfa.py:65 on the whole of ``sd``.  Reads ``second_order_tensor``, ``bc``, optional
        ``mpfa_eta`` and ``ambient_dimension``; returns the six matrices of mpfa.py:496-508."""
        k = params["second_order_tensor"]
        bc = params["bc"]
        if sd.dim <= 1:
            # mpfa.py:687-722: the scheme reduces to TPFA on a line; a point grid has no faces
            sub = {"bc": bc, "second_order_tensor": k, "ambient_dimension": params.get("ambient_dimension", sd.dim)}
            tp = Tpfa(self.keyword)
            out = tp._discretize_grid(sd, sub)
            self.last_timing = tp.last_timing
            return out
        eta = params.get("mpfa_eta", None)
        if eta is None:
            eta = determine_eta(sd)
        if np.asarray(eta).size != 1:
            raise NotImplementedError("sub-face valued mpfa_eta is not supported")
        amb = int(params.get("ambient_dimension", sd.dim))
        if amb != sd.dim and not (sd.dim == 2 and amb == 3):
            raise NotImplementedError(f"ambient_dimension={amb} for a {sd.dim}-d grid is not supported")
        if np.asarray(bc.is_dir).shape[-1] != sd.num_faces:
            raise NotImplementedError("sub-face boundary conditions are not supported")
        self._check_unsupported(params, sd)
        t0 = time.perf_counter()
        plan = DevicePlan.for_grid(sd)
        codes = scalar_bc_codes(bc, sd.num_faces)
        robw = np.asarray(bc.robin_weight, float) if np.any(codes == _lib.BC_ROB) else None
        t1 = time.perf_counter()
        kvals = k.values
        if plan.rotation is not None:  # fracture plane: mpfa.py:733-754
            kvals = rotate_second_order(kvals, plan.rotation)
        plan.mpfa_upload(kvals, codes, robw, float(np.asarray(eta).ravel()[0]))
        t2 = time.perf_counter()
        ms = plan.mpfa_assemble()
        t3 = time.perf_counter()
        # device-resident results: scipy-compatible matrices whose arrays are fetched on first touch
        out = plan.mpfa_lazy() if hasattr(plan, "mpfa_lazy") else plan.mpfa_download()
        if sd.dim == 2 and (amb == 3 or plan.rotation is not None):
            # vector source back to the ambient space, mpfa.py:423-466 (with ambient_dimension = 2 on a tilted
            # plane the reference keeps the first two ambient components, mpfa.py:459-462)
            rows = (np.eye(3) if plan.rotation is None else plan.rotation)[:2, :amb]
            for key in (self.vector_source_matrix_key, self.bound_pressure_vector_source_matrix_key):
                out[key] = _lifted(plan, out[key], rows, sd.num_cells)
        t4 = time.perf_counter()
        self.last_timing = dict(plan_s=t1 - t0, upload_s=t2 - t1, kernel_ms=ms,
                                assemble_s=t3 - t2, download_s=t4 - t3)
        _log_throughput("Mpfa", self.keyword, sd, ms, t4 - t0, out)
        return out

    def assemble_matrix_rhs(self, sd, data: dict):
        """fv_elliptic.py:67-112: A = div @ flux, b = -div @ bound_flux @ bc_values
        (- div @ vector_source_discr @ vector_source).  When the stored matrices are still device resident
        (``LazyCsr`` not yet touched) the products run on the GPU from exactly those matrices and ``A`` comes back
        as a ``LazyCsr`` backed by the device system (``A.device_csr`` feeds ``porepy_b200.krylov`` directly);
        otherwise the host scipy products of the reference."""
        mats = data[DISCRETIZATION_MATRICES][self.keyword]
        params = data[PARAMETERS][self.keyword]
        flux, bflux = mats[self.flux_matrix_key], mats[self.bound_flux_matrix_key]
        vsd = mats.get(self.vector_source_matrix_key) if "vector_source" in params else None
        if _on_device(flux, bflux) and (vsd is None or _on_device(vsd)) and flux.shape == (sd.num_faces, sd.num_cells):
            plan = flux.plan
            vec = None
            if vsd is not None:
                vec = np.asarray(params["vector_source"], dtype=np.float64)
                rows = vsd.__dict__.get("plane_rows")
                if rows is not None:  # fracture plane: the device values live in the plane's frame
                    vec = (vec.reshape(-1, rows.shape[1]) @ rows.T).ravel()
            a = plan.mpfa_system(flux.device_values)
            b = plan.mpfa_rhs(params["bc_values"], vec, bound_flux=bflux.device_values,
                              vector_source_discr=None if vsd is None else vsd.device_values)
            return _lazy_system(a), b
        div = sd.divergence(dim=1)
        matrix = div @ flux
        rhs = -div @ (bflux @ params["bc_values"])
        if "vector_source" in params:
            rhs -= div @ (mats[self.vector_source_matrix_key] @ params["vector_source"])
        return matrix, rhs

    def assemble_matrix_rhs_device(self, sd, data: dict):
        """(``DeviceCsr``, host rhs) of ``assemble_matrix_rhs``; raises unless the stored matrices are still device
        resident."""
        a, b = self.assemble_matrix_rhs(sd, data)
        if getattr(a, "device_csr", None) is None:
            raise RuntimeError("the discretization matrices are no longer device resident")
        return a.device_csr, b


class Mpsa(_Base):
    """MPSA-W stress discretization; see module docstring.  Matrix keys as mpsa.py:82-95."""

    def __init__(self, keyword: str) -> None:
        super().__init__(keyword)
        self.stress_matrix_key = "stress"
        self.bound_stress_matrix_key = "bound_stress"
        self.bound_displacement_cell_matrix_key = "bound_displacement_cell"
        self.bound_displacement_face_matrix_key = "bound_displacement_face"

    def ndof(self, sd) -> int:
        return sd.dim * sd.num_cells

    def _alphas(self, sd, params):
        return {}

    _eta_key = "mpsa_eta"

    def _discretize_grid(self, sd, params: dict) -> dict:
        """mpsa.py:121 (and biot.py:247 through ``_alphas``) on the whole of ``sd``.  Reads
        ``fourth_order_tensor``, ``bc`` (vectorial), optional ``mpsa_eta``."""
        constit = params["fourth_order_tensor"]
        bc = params["bc"]
        if getattr(bc, "bc_type", "vectorial") != "vectorial":
            raise AttributeError("MPSA must be given a vectorial boundary condition")  # mpsa.py:658
        if sd.dim == 1:
            # mpsa.py:666-697: TPFA with the longitudinal modulus 2 mu + lambda, Neumann everywhere
            if np.any(bc.is_dir):
                raise ValueError("have not considered Dirichlet boundary values here")
            from .params import BoundaryCondition, SecondOrderTensor
            tp = Tpfa("tpfa_elasticity")
            sub = {"bc": BoundaryCondition(sd), "second_order_tensor": SecondOrderTensor(2 * constit.mu + constit.lmbda)}
            t = tp._discretize_grid(sd, sub)
            return {"stress": t["flux"], "bound_stress": t["bound_flux"],
                    "bound_displacement_cell": t["bound_pressure_cell"],
                    "bound_displacement_face": t["bound_pressure_face"]}
        eta = params.get("mpsa_eta", None)
        if eta is None:
            eta = determine_eta(sd)
        hf_eta = params.get("reconstruction_eta", None)
        if hf_eta is not None and hf_eta != eta:
            raise NotImplementedError("reconstruction_eta != mpsa_eta is not supported")
        if np.asarray(bc.is_dir).shape[-1] != sd.num_faces:
            raise NotImplementedError("sub-face boundary conditions are not supported")
        self._check_unsupported(params, sd)
        alphas = self._alphas(sd, params)
        t0 = time.perf_counter()
        plan = DevicePlan.for_grid(sd)
        if plan.rotation is not None:
            # the reference discretizes in the local frame of map_grid without rotating the stiffness
            # back (mpsa.py:2005-2040): frame dependent, and not a use case (mechanics lives on the
            # top-dimensional grid)
            raise NotImplementedError("MPSA on a 2-D grid outside the xy-plane is not supported")
        codes, robw = vector_bc_codes(bc, sd.dim, sd.num_faces)
        t1 = time.perf_counter()
        plan.mpsa_upload(constit.values, codes, robw, float(eta), list(alphas.values()))
        plan.mpsa_set_basis(vector_bc_basis(bc, sd.dim, codes))
        t2 = time.perf_counter()
        ms = plan.mpsa_assemble()
        t3 = time.perf_counter()
        lazy = hasattr(plan, "mpsa_lazy")
        out = plan.mpsa_lazy() if lazy else plan.mpsa_download()
        if alphas:
            coupled = {k: {} for k in ("displacement_divergence", "boundary_displacement_divergence",
                                       "scalar_gradient", "mpsa_consistency",
                                       "bound_displacement_pressure")}
            for q, key in enumerate(alphas):
                for name, m in (plan.biot_lazy(q) if lazy else plan.biot_download(q)).items():
                    coupled[name][key] = m
            out.update(coupled)
        t4 = time.perf_counter()
        self.last_timing = dict(plan_s=t1 - t0, upload_s=t2 - t1, kernel_ms=ms,
                                assemble_s=t3 - t2, download_s=t4 - t3)
        _log_throughput(type(self).__name__, self.keyword, sd, ms, t4 - t0, out)
        return out

    def assemble_matrix_rhs(self, sd, data: dict):
        """mpsa.py:486-529; device path as in ``Mpfa.assemble_matrix_rhs``."""
        mats = data[DISCRETIZATION_MATRICES][self.keyword]
        params = data[PARAMETERS][self.keyword]
        stress, bstress = mats["stress"], mats["bound_stress"]
        if _on_device(stress, bstress) and stress.shape[0] == sd.num_faces * sd.dim:
            plan = stress.plan
            a = plan.mpsa_system(stress.device_values)
            b = plan.mpsa_rhs(params["bc_values"], params["source"], bound_stress=bstress.device_values)
            return _lazy_system(a), b
        div = sd.divergence(dim=sd.dim)
        matrix = div @ stress
        rhs = -div @ (bstress @ params["bc_values"]) + params["source"]
        return matrix, rhs

    def assemble_matrix_rhs_device(self, sd, data: dict):
        """(``DeviceCsr``, host rhs); see ``Mpfa.assemble_matrix_rhs_device``."""
        a, b = self.assemble_matrix_rhs(sd, data)
        if getattr(a, "device_csr", None) is None:
            raise RuntimeError("the discretization matrices are no longer device resident")
        return a.device_csr, b


class Biot(Mpsa):
    """MPSA + Biot coupling terms (biot.py:40; keys :94-111, dict-valued per coupling keyword)."""

    def __init__(self, keyword: str = "mechanics") -> None:
        super().__init__(keyword)
        self.displacement_divergence_matrix_key = "displacement_divergence"
        self.bound_displacement_divergence_matrix_key = "boundary_displacement_divergence"
        self.scalar_gradient_matrix_key = "scalar_gradient"
        self.consistency_matrix_key = "mpsa_consistency"
        self.bound_pressure_matrix_key = "bound_displacement_pressure"

    def _alphas(self, sd, params):
        out = {}
        for key, a in params["scalar_vector_mappings"].items():
            if isinstance(a, (float, int, np.floating, np.integer)):
                v = np.zeros((3, 3, sd.num_cells))
                v[0, 0] = v[1, 1] = v[2, 2] = float(a)  # biot.py:312-321
            else:
                v = np.asarray(a.values, float)
            out[key] = v
        if len(out) > 4:
            raise NotImplementedError("at most 4 coupling tensors per Biot discretization")
        return out

    def assemble_matrix_rhs(self, sd, data: dict):
        """biot.py:125-149."""
        raise NotImplementedError("This class cannot be used for assembly.\nUse the ad version instead")


def _empty_flux_terms(discr, sd, vdim: int) -> dict:
    """The 0-D shortcut of tpfa.py:87-104 (a point grid has no faces)."""
    nc = sd.num_cells
    return {
        discr.flux_matrix_key: sps.csr_matrix((0, nc)),
        discr.bound_flux_matrix_key: sps.csr_matrix((0, 0)),
        discr.bound_pressure_cell_matrix_key: sps.csr_matrix((0, nc)),
        discr.bound_pressure_face_matrix_key: sps.csr_matrix((0, 0)),
        discr.vector_source_matrix_key: sps.csr_matrix((0, nc * max(vdim, 1))),
        discr.bound_pressure_vector_source_matrix_key: sps.csr_matrix((0, nc * max(vdim, 1))),
    }


class Tpfa(Mpfa):
    """Two-point flux approximation (numerics/fv/tpfa.py:18; same keys and ``assemble_matrix_rhs`` as
    MPFA through FVElliptic).  One thread per face on a ``FaceGrid``; grids of any dimension, anywhere in
    space (the reference works on the 3-D coordinates, tpfa.py:160-175)."""

    def discretize(self, sd, data: dict) -> None:
        """tpfa.py:40: always the whole grid -- the reference's TPFA has no partial mode, so
        ``specified_cells/faces/nodes`` (possibly left behind by an MPFA update on the same keyword,
        _fvutils.py:346-353) and ``update_discretization`` are ignored."""
        params = data[PARAMETERS][self.keyword]
        mats = data.setdefault(DISCRETIZATION_MATRICES, {}).setdefault(self.keyword, {})
        mats.update(self._discretize_grid(sd, params))

    def _discretize_grid(self, sd, params: dict) -> dict:
        vdim = int(params.get("ambient_dimension", sd.dim))
        if sd.dim == 0:
            return _empty_flux_terms(self, sd, vdim)
        k = params["second_order_tensor"]
        bc = params["bc"]
        self._check_unsupported(params, sd)
        t0 = time.perf_counter()
        fg = FaceGrid.for_grid(sd)
        fc = sps.csr_matrix(sd.cell_faces)
        fc.sort_indices()
        ip, ix = fc.indptr, fc.indices
        vals = fg.tpfa(k.values, face_bc_bits(bc, sd.num_faces), ip, vdim)
        nf, nc = sd.num_faces, sd.num_cells
        boundary = np.diff(ip) == 1
        cols_v = (ix[:, None].astype(np.int64) * vdim + np.arange(vdim)).ravel()
        ipv = ip.astype(np.int64) * vdim
        self.last_timing = dict(total_s=time.perf_counter() - t0)
        return {
            self.flux_matrix_key: sps.csr_matrix((vals[0], ix, ip), shape=(nf, nc)),
            self.bound_flux_matrix_key: sps.diags(np.where(boundary, vals[4], 0.0)).tocsr(),
            self.bound_pressure_cell_matrix_key: sps.csr_matrix((vals[1], ix, ip), shape=(nf, nc)),
            self.bound_pressure_face_matrix_key: sps.diags(vals[5]).tocsr(),
            self.vector_source_matrix_key: sps.csr_matrix((vals[2], cols_v, ipv), shape=(nf, nc * vdim)),
            self.bound_pressure_vector_source_matrix_key: sps.csr_matrix((vals[3], cols_v, ipv),
                                                                         shape=(nf, nc * vdim)),
        }


class Upwind(_Base):
    """First-order upwinding of an advective flux (numerics/fv/upwind.py:13).  ``discretize`` reads
    ``bc`` and the face fluxes under ``flux_array_key`` (default ``"darcy_flux"``) and writes the
    upwind matrix and the two boundary matrices; ``assemble_matrix_rhs`` as upwind.py:57-148."""

    def __init__(self, keyword: str = "transport") -> None:
        super().__init__(keyword)
        self.upwind_matrix_key = "transport"
        self.bound_transport_dir_matrix_key = "rhs_dir"
        self.bound_transport_neu_matrix_key = "rhs_neu"
        self._flux_array_key = "darcy_flux"

    @property
    def flux_array_key(self) -> str:
        return self._flux_array_key

    @flux_array_key.setter
    def flux_array_key(self, value: str) -> None:
        self._flux_array_key = value

    def ndof(self, sd) -> int:
        return sd.num_cells

    def discretize(self, sd, data: dict) -> None:
        params = data[PARAMETERS][self.keyword]
        mats = data.setdefault(DISCRETIZATION_MATRICES, {}).setdefault(self.keyword, {})
        bc = params.get("bc")
        if bc is None:  # upwind.py:244-247: Dirichlet on the boundary
            from .params import BoundaryCondition
            bc = BoundaryCondition(sd, sd.get_boundary_faces(), "dir")
        nf, nc = sd.num_faces, sd.num_cells
        ncomp = int(params.get("num_components", 1))
        if nf == 0:  # point grids: upwind.py:226-236
            mats[self.upwind_matrix_key] = sps.csr_matrix((0, nc * ncomp))
            mats[self.bound_transport_neu_matrix_key] = sps.csr_matrix((0, 0))
            mats[self.bound_transport_dir_matrix_key] = sps.csr_matrix((0, 0))
            return
        fg = FaceGrid.for_grid(sd)
        bits = face_bc_bits(bc, nf)
        up, neu, dr = fg.upwind(params[self._flux_array_key], bits)
        # A boundary face that is neither Dirichlet nor Neumann (Robin / unflagged) with inflow has no upstream
        # cell: the reference ends up with column index -1 and scipy raises (upwind.py:272-281).  Fail as loudly.
        single = np.diff(sps.csr_matrix(sd.cell_faces).indptr) == 1
        orphan = single & (up < 0) & ((bits & 12) == 0)
        if orphan.any():
            raise ValueError(f"upwind: boundary face {int(np.flatnonzero(orphan)[0])} has inflow but neither a "
                             "Dirichlet nor a Neumann condition")
        rows = np.flatnonzero(up >= 0)
        m = sps.csr_matrix((np.ones(rows.size), (rows, up[rows])), shape=(nf, nc))
        eye = sps.eye(ncomp)
        mats[self.upwind_matrix_key] = sps.kron(m, eye).tocsr()
        mats[self.bound_transport_neu_matrix_key] = sps.kron(sps.diags(neu), eye).tocsr()
        mats[self.bound_transport_dir_matrix_key] = sps.kron(sps.diags(dr), eye).tocsr()

    def assemble_matrix_rhs(self, sd, data: dict):
        """upwind.py:57-148: ``div @ diag(q) @ upwind`` and the boundary right-hand side."""
        mats = data[DISCRETIZATION_MATRICES][self.keyword]
        params = data[PARAMETERS][self.keyword]
        q = sps.diags(np.asarray(params[self._flux_array_key], float))
        div = sd.divergence(dim=1)
        if div.shape[1] != mats[self.upwind_matrix_key].shape[0]:
            raise ValueError("Dimension mismatch: upwinding with several components is only supported in Ad mode")
        matrix = div @ q @ mats[self.upwind_matrix_key]
        rhs = div @ ((mats[self.bound_transport_neu_matrix_key] + mats[self.bound_transport_dir_matrix_key] @ q)
                     @ params["bc_values"])
        return matrix, rhs


def interface_upwind_masks(interface_flux):
    """(sign, upstream-is-primary, upstream-is-secondary) per mortar cell through ``pb_upwind_coupling`` (one thread per
    entry).  A separate function so that the CPU tests can substitute the host formulas."""
    lam = _lib.f64(interface_flux)
    lib = _lib.load()
    _lib.require_gpu()
    n = int(lam.size)
    sgn, up1, up2 = np.empty(n), np.empty(n), np.empty(n)
    _lib.check(lib.pb_upwind_coupling(n, _lib.ptr(lam, _lib._f64p), _lib.ptr(sgn, _lib._f64p),
                                      _lib.ptr(up1, _lib._f64p), _lib.ptr(up2, _lib._f64p)))
    return sgn, up1, up2


class UpwindCoupling:
    """Upwinding of an advective flux across the interface between a subdomain and a lower-dimensional one
    (numerics/fv/upwind.py:377).  ``discretize`` writes the reference's six matrices to
    ``data_intf["discretization_matrices"][keyword]``; ``assemble_matrix_rhs`` as upwind.py:530-680."""

    def __init__(self, keyword: str) -> None:
        self.keyword = keyword
        self.trace_primary_matrix_key = "trace"
        self.inv_trace_primary_matrix_key = "inv_trace"
        self.upwind_primary_matrix_key = "upwind_primary"
        self.upwind_secondary_matrix_key = "upwind_secondary"
        self.flux_matrix_key = "flux"
        self.mortar_discr_matrix_key = "mortar_discr"
        self._flux_array_key = "darcy_flux"

    def key(self) -> str:
        return self.keyword + "_"

    def discretization_key(self):
        return self.key() + DISCRETIZATION_MATRICES

    @property
    def flux_array_key(self) -> str:
        return self._flux_array_key

    @flux_array_key.setter
    def flux_array_key(self, value: str) -> None:
        self._flux_array_key = value

    def ndof(self, intf) -> int:
        return intf.num_cells

    def discretize(self, sd_primary, sd_secondary, intf, data_primary, data_secondary, data_intf) -> None:
        if sd_primary.dim - sd_secondary.dim not in [1, 2]:
            raise ValueError("Implementation is only valid for grids one dimension apart.")
        mats = data_intf.setdefault(DISCRETIZATION_MATRICES, {}).setdefault(self.keyword, {})
        sgn, up1, up2 = interface_upwind_masks(data_intf[PARAMETERS][self.keyword][self._flux_array_key])
        inv_trace = abs(sd_primary.divergence(dim=1))
        mats[self.inv_trace_primary_matrix_key] = inv_trace
        mats[self.trace_primary_matrix_key] = inv_trace.T
        mats[self.upwind_primary_matrix_key] = sps.diags(up1)
        mats[self.upwind_secondary_matrix_key] = sps.diags(up2)
        mats[self.flux_matrix_key] = sps.diags(sgn)
        mats[self.mortar_discr_matrix_key] = sps.eye(intf.num_cells)

    def assemble_matrix_rhs(self, sd_primary, sd_secondary, intf, data_primary, data_secondary, data_intf, matrix):
        """upwind.py:530-680: the 3 x 3 block contribution of the coupling condition (right-hand side zero)."""
        m = data_intf[DISCRETIZATION_MATRICES][self.keyword]
        dof = np.array([matrix[0, 0].shape[1], matrix[1, 1].shape[1], intf.num_cells])
        cc = np.array([sps.coo_matrix((i, j)) for i in dof for j in dof]).reshape((3, 3))
        lam = np.abs(data_intf[PARAMETERS][self.keyword][self._flux_array_key])
        scaling = sps.dia_matrix((lam, 0), shape=(intf.num_cells, intf.num_cells))
        cc[0, 2] = m[self.inv_trace_primary_matrix_key] @ intf.mortar_to_primary_int()
        cc[1, 2] = -intf.mortar_to_secondary_int()
        cc[2, 0] = (scaling @ m[self.flux_matrix_key] @ m[self.upwind_primary_matrix_key]
                    @ intf.primary_to_mortar_avg() @ m[self.trace_primary_matrix_key])
        cc[2, 1] = scaling @ m[self.flux_matrix_key] @ m[self.upwind_secondary_matrix_key] @ intf.secondary_to_mortar_avg()
        cc[2, 2] = -m[self.mortar_discr_matrix_key]
        if sd_primary == sd_secondary:
            cc = np.array([np.sum(cc, axis=(0, 1))])
        rhs = np.array([np.zeros(dof[0]), np.zeros(dof[1]), np.zeros(dof[2])], dtype=object)
        if rhs.ndim == 2:
            rhs = rhs.ravel()
        matrix += cc
        return matrix, rhs
