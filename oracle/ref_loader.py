"""Import the unmodified PorePy reference: from ``/root/reference/src`` (build container) or from the copy
``oracle/_ref`` that ``oracle/make_ref.sh`` places next to this file (git-ignored, shipped to the GPU box like
the built ``.so`` files; the reference is pure Python, so "building" it is a copy).

TEST / BASELINE INFRASTRUCTURE ONLY: used by tools/make_golden.py, tools/make_digests.py, the "reference
present" tests, and by ``bench.py --impl reference`` / ``cpu_baseline`` to time ``pp.Mpfa.discretize`` +
``pp.Mpsa.discretize`` on the bench box's host cores.  The product (porepy_b200/) never imports this.
Third-party modules the hot path never touches and that are absent from the image are stubbed before
``import porepy`` (SURVEY.md 8c).
"""
from __future__ import annotations

import os
import sys
import types
from unittest.mock import MagicMock

_HERE = os.path.dirname(os.path.abspath(__file__))
_CANDIDATES = ["/root/reference/src", os.path.join(_HERE, "_ref")]
REF_SRC = next((p for p in _CANDIDATES if os.path.isdir(os.path.join(p, "porepy"))), _CANDIDATES[0])
# the reference's own test suite: next to src/ in the reference tree, inside the copy under oracle/_ref
REF_TESTS = next((p for p in (os.path.join(os.path.dirname(REF_SRC), "tests"), os.path.join(REF_SRC, "tests"))
                  if os.path.isdir(p)), None)

_STUBS = [
    "meshio", "gmsh", "shapely", "shapely.geometry", "shapely.speedups",
    "matplotlib", "matplotlib.pyplot", "matplotlib.colors", "matplotlib.tri",
    "matplotlib.patches", "matplotlib.figure", "matplotlib.axes",
    "matplotlib.ticker", "matplotlib.lines", "matplotlib.collections",
    "matplotlib.cm", "matplotlib.animation", "mpl_toolkits",
    "mpl_toolkits.mplot3d", "mpl_toolkits.mplot3d.art3d",
    "mpl_toolkits.axes_grid1", "deepdiff", "seaborn", "future",
]


class _Stub(types.ModuleType):
    __path__: list = []

    def __getattr__(self, name):
        if name.startswith("__") and name.endswith("__"):
            raise AttributeError(name)
        return MagicMock()


REF_MAX_THREADS = 32


def _cap_numba_threads() -> None:
    """The reference inverts its local systems inside a numba ``prange`` (``invert_diagonal_blocks``,
    matrix_operations.py:1310-1371); every numba thread calls LAPACK.  The image's OpenBLAS supports at most 128
    calling threads and aborts ("too many memory regions") on the GPU boxes, whose hosts have more cores than
    that.  Cap the pool at ``REF_MAX_THREADS`` (the inversion is memory bound: more threads measured slower)."""
    n = max(1, min(os.cpu_count() or 1, REF_MAX_THREADS))
    if "numba" not in sys.modules:
        os.environ.setdefault("NUMBA_NUM_THREADS", str(n))
    try:
        import numba
        numba.set_num_threads(min(n, numba.config.NUMBA_NUM_THREADS))
    except Exception:
        pass


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REF_SRC, "porepy"))


def load_porepy():
    """Return the reference ``porepy`` module, or raise ImportError."""
    if "porepy" in sys.modules:
        return sys.modules["porepy"]
    if not reference_available():
        raise ImportError("reference not present: neither /root/reference/src nor oracle/_ref (run oracle/make_ref.sh)")
    for name in _STUBS:
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:
                sys.modules[name] = _Stub(name)
    if REF_SRC not in sys.path:
        sys.path.insert(0, REF_SRC)
    _cap_numba_threads()
    import porepy  # noqa: E402
    _cap_numba_threads()

    return porepy


def reference_grid(pp, g):
    """``pp.Grid`` with the topology and geometry arrays of the porepy_b200 grid ``g`` (the discretizations read
    only these arrays and the signs of ``cell_faces``; the reference's ``compute_geometry`` is not needed)."""
    import numpy as np
    import scipy.sparse as sps
    name = "StructuredTetrahedralGrid" if "Tetrahedral" in str(g.name) else (
        "StructuredTriangleGrid" if "Triangle" in str(g.name) else "CartGrid")
    r = pp.Grid(int(g.dim), np.array(g.nodes), sps.csc_matrix(g.face_nodes), sps.csc_matrix(g.cell_faces), name)
    for attr in ("face_normals", "face_centers", "face_areas", "cell_centers", "cell_volumes"):
        setattr(r, attr, np.array(getattr(g, attr)))
    return r


def reference_discretize(pp, g, k, bc, C, vbc, alpha=None):
    """``pp.Mpfa("flow").discretize`` + ``pp.Mpsa("mech").discretize`` (``pp.Biot`` with ``alpha``) of the unmodified
    reference on the porepy_b200 grid / parameter objects.  Returns (seconds_mpfa, seconds_mpsa, data_flow, data_mech)."""
    import time
    r = reference_grid(pp, g)
    rbc = pp.BoundaryCondition(r)
    rbc.is_dir, rbc.is_neu, rbc.is_rob = bc.is_dir.copy(), bc.is_neu.copy(), bc.is_rob.copy()
    rk = pp.SecondOrderTensor(k.values[0, 0].copy())
    rk.values = k.values.copy()
    d1 = pp.initialize_data({}, "flow", {"second_order_tensor": rk, "bc": rbc})
    t0 = time.perf_counter()
    pp.Mpfa("flow").discretize(r, d1)
    t1 = time.perf_counter()
    rvbc = pp.BoundaryConditionVectorial(r)
    rvbc.is_dir, rvbc.is_neu, rvbc.is_rob = vbc.is_dir.copy(), vbc.is_neu.copy(), vbc.is_rob.copy()
    rC = pp.FourthOrderTensor(C.mu.copy(), C.lmbda.copy())
    prm = {"fourth_order_tensor": rC, "bc": rvbc}
    cls = pp.Mpsa
    if alpha is not None:
        ra = pp.SecondOrderTensor(alpha.values[0, 0].copy())
        ra.values = alpha.values.copy()
        prm["scalar_vector_mappings"] = {"flow": ra}
        cls = pp.Biot
    d2 = pp.initialize_data({}, "mech", prm)
    t2 = time.perf_counter()
    cls("mech").discretize(r, d2)
    t3 = time.perf_counter()
    return t1 - t0, t3 - t2, d1, d2
