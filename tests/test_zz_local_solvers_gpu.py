"""The dense interaction-region solvers on the device, configuration by configuration, against an extended-precision
reference (tests/local_solver_cases.py), and the assembly's use of every configuration against the oracle.

Solver part: every configuration 0..7, with the matrix in shared memory and in the global-memory workspace, at the
sizes where blocked kernels go wrong (every remainder mod 4, the neighbours of every multiple of 8, the largest
order), one right-hand side and as many as fill the configuration's width.  Families drive the fast and the slow
pivoting paths of the blocked solver, the growth threshold between them and column-graded panels.  Bound:
max|X - X_ref| / max|X_ref| <= 50 n u kappa_inf(M).

Assembly part: a table of grids and discretizations whose class report must contain given configurations; the
union of the reports must reach all eight configurations and both places of the matrix."""
import os

import numpy as np
import pytest

import local_solver_cases as lc
import porepy_b200 as pb
from cases import flatten, max_rel_err
from porepy_b200.fv import NUM_SOLVER_CFGS, local_solve_batch, solver_limits

pytestmark = pytest.mark.gpu

WIDE = 256          # right-hand-side columns generated per order; a run takes the first nrhs
CFG6_EXTRA = (127, 128, 129, 160, 199, 200)   # the catch-all configuration beyond the blocked solvers' orders
_CASES = {}


def _cases(n):
    """[(family, M sent to the solver, d, X_ref, kappa)]: d * X(M) is compared with X_ref (d = 1 except for family
    C, whose reference is the system before the column grading)."""
    if n in _CASES:
        return _CASES[n]
    B = lc.rhs(n, WIDE)
    out = []

    def add(fam, M, Mu=None, d=None):
        Mu = M if Mu is None else Mu
        d = np.ones(n) if d is None else d
        out.append((fam, M, d, lc.ref_solve(Mu, B, iters=3), lc.cond_inf(Mu)))

    add("F", lc.family_f(n))
    if n >= 8:
        add("S", lc.family_s(n))
    for seed in (0, 1):
        add("M", lc.family_m_gauss(n, seed))
    Q = (n + 3) // 4
    for k in sorted({0, Q // 2, Q - 1}):
        if n - 4 * k >= 2:
            add("M", lc.family_m_panel(n, k))
    if n >= 2:
        for target, _ in lc.G_TARGETS:
            add("G", lc.family_g(n, target))
    for e in lc.C_EXPONENTS:
        M, Mu, d = lc.family_c(n, e)
        add(f"C{e}", M, Mu, d)
    _CASES[n] = (B, out)
    return _CASES[n]


def _orders(cfg):
    _, max_n, _ = solver_limits(cfg)
    if cfg == 6:
        return lc.sizes(112) + list(CFG6_EXTRA)
    return lc.sizes(max_n)


def _widths(cfg, n):
    _, _, max_w = solver_limits(cfg)
    top = WIDE if cfg == 6 else max_w
    return sorted({1, top - n} - {0}) if top - n >= 1 else []


def _solve(cfg, A, n, a_global):
    """None when the matrix does not fit the shared memory (the assembly then puts it in the workspace)."""
    try:
        return local_solve_batch(cfg, A, n, a_global)
    except ValueError as e:
        if not a_global and "shared memory" in str(e):
            return None
        raise


def test_limits_match_the_class_table():
    lim = [solver_limits(c) for c in range(NUM_SOLVER_CFGS)]
    assert lim[6][1] == lim[6][2] == 2**31 - 1
    for c in (0, 1, 2, 3, 4, 5, 7):
        team, mn, mw = lim[c]
        assert team % 32 == 0 and 1 <= mn <= 255 and mn < mw
    with pytest.raises(ValueError):
        solver_limits(8)
    # sizes beyond a configuration are refused before any launch
    team, mn, mw = lim[0]
    with pytest.raises(ValueError):
        local_solve_batch(0, np.zeros((1, mn + 1, mn + 2)), mn + 1)
    with pytest.raises(ValueError):
        local_solve_batch(0, np.zeros((1, 4, mw + 1)), 4)


@pytest.mark.parametrize("cfg", range(NUM_SOLVER_CFGS))
def test_solver_accuracy(cfg, capsys):
    worst, bad, ran = {}, [], {0: 0, 1: 0}
    for a_global in (0, 1):
        for n in _orders(cfg):
            B, cases = _cases(n)
            for nrhs in _widths(cfg, n):
                A = np.stack([np.hstack([M, B[:, :nrhs]]) for _, M, _, _, _ in cases])
                res = _solve(cfg, A, n, a_global)
                if res is None:
                    continue
                ran[a_global] += 1
                X, ok = res
                for (fam, M, d, Xref, kappa), x, good in zip(cases, X, ok):
                    r = lc.error_ratio(d[:, None] * x, Xref[:, :nrhs], M, kappa) if good else np.inf
                    key = (fam[0] if fam[0] != "C" else fam)
                    worst[key] = max(worst.get(key, 0.0), r)
                    if not good or not r <= 1.0:
                        bad.append((a_global, n, nrhs, fam, bool(good), r))
    with capsys.disabled():
        print(f"\ncfg {cfg}: worst err / (50 n u kappa) per family: "
              + ", ".join(f"{k} {v:.2e}" for k, v in sorted(worst.items()))
              + f"  (runs: shared {ran[0]}, workspace {ran[1]})")
        if bad:
            print(f"cfg {cfg}: {len(bad)} failures (a_global, n, nrhs, family, ok, ratio), first 20:", bad[:20])
    assert ran[0] > 0 and ran[1] > 0
    assert not bad, f"cfg {cfg}: {len(bad)} systems refused or outside the bound, e.g. {bad[:8]}"


def _singular_cases(n):
    out = [("duplicate_row", lc.singular_duplicate_row(n)), ("zero_column", lc.singular_zero_column(n))]
    if n % 4 == 3:
        out.append(("last_panel", lc.singular_last_panel(n)))
    return out


def _refusal_orders(cfg):
    _, max_n, _ = solver_limits(cfg)
    top = 200 if cfg == 6 else max_n
    return sorted({n for n in (2, 3, 4, 5, 7, 8, 11, 15, 16, 31, 33, 47, 48, 111, 112, top - 1, top)
                   if 2 <= n <= top})


@pytest.mark.parametrize("cfg", range(NUM_SOLVER_CFGS))
def test_singular_and_nonfinite_systems(cfg):
    _, _, max_w = solver_limits(cfg)
    for a_global in (0, 1):
        for n in _refusal_orders(cfg):
            nrhs = min(3, (WIDE if cfg == 6 else max_w) - n)
            if nrhs < 1:
                continue
            B = lc.rhs(n, nrhs)
            sing = _singular_cases(n)
            nonf = [("nan", lc.nonfinite(n, "nan")), ("inf", lc.nonfinite(n, "inf"))]
            A = np.stack([np.hstack([M, B]) for _, M in sing + nonf])
            res = _solve(cfg, A, n, a_global)
            if res is None:
                continue
            X, ok = res
            for (name, _), good in zip(sing, ok[:len(sing)]):
                assert not good, (cfg, a_global, n, name)
            for (name, _), good, x in zip(nonf, ok[len(sing):], X[len(sing):]):
                assert not (good and np.all(np.isfinite(x))), (cfg, a_global, n, name)
                assert not good, (cfg, a_global, n, name)   # every configuration refuses non-finite systems


@pytest.mark.parametrize("cfg", range(NUM_SOLVER_CFGS))
def test_batch_isolation(cfg):
    """Teams do not see each other: the same system in every slot gives the same bits; a refused system leaves the
    bits of its neighbours unchanged; part-filled CTAs (4q+1, 4q+3 systems) and batches beyond the resident teams
    (grid-stride loop, workspace reuse) change nothing, and neither does the place of the matrix."""
    n, nrhs = 5, 3
    good = np.hstack([lc.family_m_gauss(n, 3), lc.rhs(n, nrhs)])
    bad = np.hstack([lc.singular_zero_column(n), lc.rhs(n, nrhs)])
    ref_bits = None
    for a_global in (0, 1):
        for nsys in (9, 11, 20001):
            A = np.repeat(good[None], nsys, axis=0)
            X, ok = local_solve_batch(cfg, A, n, a_global)
            assert ok.all()
            assert np.array_equal(X.view(np.int64), np.broadcast_to(X[0], X.shape).view(np.int64))
            if ref_bits is None:
                ref_bits = X[0].copy()
            assert np.array_equal(X[0].view(np.int64), ref_bits.view(np.int64))
            for k in sorted({0, 1, nsys // 2, nsys - 2, nsys - 1}):
                A2 = A.copy()
                A2[k] = bad
                X2, ok2 = local_solve_batch(cfg, A2, n, a_global)
                assert not ok2[k] and np.all(np.isnan(X2[k]))
                keep = np.arange(nsys) != k
                assert ok2[keep].all()
                assert np.array_equal(X2[keep].view(np.int64), X[keep].view(np.int64))


def test_configurations_agree():
    """Systems that fit every configuration: the same result from each, within the bound, and the same verdict on
    singular and non-finite systems."""
    lims = [solver_limits(c) for c in range(NUM_SOLVER_CFGS)]
    max_n = min(m for _, m, _ in lims)
    max_w = min(w for _, _, w in lims)
    for n in (1, 2, 3, 5, 8, 12, max_n):
        B, cases = _cases(n)
        for nrhs in (1, max_w - n):
            A = np.stack([np.hstack([M, B[:, :nrhs]]) for _, M, _, _, _ in cases])
            Xs = [local_solve_batch(c, A, n)[0] for c in range(NUM_SOLVER_CFGS)]
            for i, (fam, M, d, Xref, kappa) in enumerate(cases):
                bound = 50.0 * n * lc.U * kappa
                scale = np.abs(Xref[:, :nrhs]).max()
                for c in range(1, NUM_SOLVER_CFGS):
                    diff = np.abs(d[:, None] * (Xs[c][i] - Xs[0][i])).max() / scale
                    assert diff <= 2 * bound, (n, nrhs, fam, c, diff / bound)
        if n >= 2:
            sing = [M for _, M in _singular_cases(n)] + [lc.nonfinite(n, "nan"), lc.nonfinite(n, "inf")]
            A = np.stack([np.hstack([M, lc.rhs(n, 2)]) for M in sing])
            oks = np.array([local_solve_batch(c, A, n)[1] for c in range(NUM_SOLVER_CFGS)])
            assert not oks.any(), (n, oks)


# ---------------------------------------------------------------------------------------------------------------------
# assembly coverage
# ---------------------------------------------------------------------------------------------------------------------
def icosahedral_ball():
    """A once-subdivided icosahedron (80 triangles) joined to its centre: 80 tetrahedra around one node, whose
    interaction region has 120 sub-faces."""
    t = (1 + 5 ** 0.5) / 2
    v = [[-1, t, 0], [1, t, 0], [-1, -t, 0], [1, -t, 0], [0, -1, t], [0, 1, t], [0, -1, -t], [0, 1, -t],
         [t, 0, -1], [t, 0, 1], [-t, 0, -1], [-t, 0, 1]]
    f = [[0, 11, 5], [0, 5, 1], [0, 1, 7], [0, 7, 10], [0, 10, 11], [1, 5, 9], [5, 11, 4], [11, 10, 2],
         [10, 7, 6], [7, 1, 8], [3, 9, 4], [3, 4, 2], [3, 2, 6], [3, 6, 8], [3, 8, 9], [4, 9, 5], [2, 4, 11],
         [6, 2, 10], [8, 6, 7], [9, 8, 1]]
    v = [np.array(x, float) / np.linalg.norm(x) for x in v]
    mid = {}

    def m(a, b):
        k = (min(a, b), max(a, b))
        if k not in mid:
            p = v[a] + v[b]
            v.append(p / np.linalg.norm(p))
            mid[k] = len(v) - 1
        return mid[k]

    tri = []
    for a, b, c in f:
        ab, bc, ca = m(a, b), m(b, c), m(c, a)
        tri += [[a, ab, ca], [b, bc, ab], [c, ca, bc], [ab, bc, ca]]
    nodes = np.array(v + [np.zeros(3)]).T
    cn = np.array([[len(v), *x] for x in tri])
    return pb.tet_grid_from_cells(nodes, cn)


def _fresh(g):
    if hasattr(g, "_b200_plan"):
        del g._b200_plan
    return g


def _aniso(nc, rng):
    return pb.SecondOrderTensor(1 + rng.random(nc), 1 + rng.random(nc), 1 + rng.random(nc),
                                0.3 * rng.random(nc), 0.3 * rng.random(nc), 0.3 * rng.random(nc))


def _scalar_bc(g, robin=False):
    bf = g.get_all_boundary_faces()
    x = g.face_centers[0, bf]
    lab = np.where(x < x.min() + 1e-10, "dir", "rob" if robin else "neu")
    return pb.BoundaryCondition(g, bf, list(lab))


def _vector_bc(g):
    bf = g.get_all_boundary_faces()
    lo = g.face_centers[0, bf] < g.face_centers[0, bf].min() + 1e-10
    return pb.BoundaryConditionVectorial(g, bf[lo], "dir")


def _run_mpfa(g, k, bc):
    from oracle import fv_oracle as fo
    data = pb.initialize_data({}, "flow", {"second_order_tensor": k, "bc": bc})
    pb.Mpfa("flow").discretize(g, data)
    err, key = max_rel_err(fo.mpfa(g, k.values, bc, pb.determine_eta(g)), data[pb.DISCRETIZATION_MATRICES]["flow"])
    return pb.DevicePlan.for_grid(g).node_classes("mpfa"), err, key


def _run_mpsa(g, C, bc, alpha):
    from oracle import fv_oracle as fo
    params = {"fourth_order_tensor": C, "bc": bc}
    if alpha:
        params["scalar_vector_mappings"] = {"flow": 0.8}
    data = pb.initialize_data({}, "mech", params)
    (pb.Biot("mech") if alpha else pb.Mpsa("mech")).discretize(g, data)
    ref = flatten(fo.mpsa(g, C.values, bc, pb.determine_eta(g), alpha={"flow": 0.8} if alpha else None))
    err, key = max_rel_err(ref, data[pb.DISCRETIZATION_MATRICES]["mech"])
    return pb.DevicePlan.for_grid(g).node_classes("mpsa"), err, key


def _stiffness(g, rng):
    nc = g.num_cells
    return pb.FourthOrderTensor(np.exp(0.3 * rng.standard_normal(nc)), np.exp(0.3 * rng.standard_normal(nc)))


def _contrast(g, rng):
    """Permeability 1e-4 or 1e4 per cell: neighbouring cells differ by up to 1e8."""
    return pb.SecondOrderTensor(np.where(rng.random(g.num_cells) < 0.5, 1e-4, 1e4))


# (name, grid, discretization, (cfg, a_global) pairs that must appear -- a_global None: either --, environment)
COVERAGE = [
    ("hex mpfa", lambda: pb.cart_grid_3d([4, 4, 3], perturb=0.25, seed=4), "mpfa", {(0, False)}, {}),
    ("hex mpsa", lambda: pb.cart_grid_3d([4, 4, 3], perturb=0.25, seed=4), "mpsa", {(1, False)}, {}),
    ("hex biot", lambda: pb.cart_grid_3d([4, 4, 3], perturb=0.25, seed=4), "biot", {(2, False)}, {}),
    ("tet mpfa", lambda: pb.structured_tet_grid([3, 3, 2]), "mpfa", {(3, False)}, {}),
    ("tet mpsa", lambda: pb.structured_tet_grid([3, 3, 2]), "mpsa", {(4, False)}, {}),
    ("tet biot", lambda: pb.structured_tet_grid([3, 3, 2]), "biot", {(5, None)}, {}),
    ("2-D mpfa", lambda: pb.cart_grid_2d([6, 5]), "mpfa", set(), {}),
    ("2-D biot", lambda: pb.cart_grid_2d([6, 5]), "biot", set(), {}),
    ("ball mpfa", icosahedral_ball, "mpfa", {(6, True)}, {}),
    ("ball mpsa", icosahedral_ball, "mpsa", {(6, True)}, {}),
    ("ball biot", icosahedral_ball, "biot", {(6, True)}, {}),
    ("tet mpsa, POREB200_CFG4=reg", lambda: pb.structured_tet_grid([3, 3, 2]), "mpsa", {(7, False)},
     {"POREB200_CFG4": "reg"}),
    ("hex mpfa, contrast 1e8, Robin", lambda: pb.cart_grid_3d([5, 4, 4], perturb=0.2, seed=6), "contrast",
     {(0, False)}, {}),
    ("tet mpfa, contrast 1e8, Robin", lambda: pb.structured_tet_grid([3, 3, 3]), "contrast", {(3, False)}, {}),
]


def test_assembly_class_coverage(capsys):
    rng = np.random.default_rng(17)
    union = set()
    rows = []
    for name, make, kind, expected, env in COVERAGE:
        g = _fresh(make())
        saved = {k: os.environ.get(k) for k in env}
        os.environ.update(env)
        try:
            if kind == "mpfa":
                cls, err, key = _run_mpfa(g, _aniso(g.num_cells, rng), _scalar_bc(g))
            elif kind == "contrast":
                cls, err, key = _run_mpfa(g, _contrast(g, rng), _scalar_bc(g, robin=True))
            else:
                cls, err, key = _run_mpsa(g, _stiffness(g, rng), _vector_bc(g), alpha=kind == "biot")
        finally:
            for k, v in saved.items():
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
            _fresh(g)
        got = {(c, a) for c, a, _ in cls}
        rows.append((name, cls, err))
        union |= got
        assert all(any(c == ce and (ae is None or a == ae) for c, a in got) for ce, ae in expected), (name, cls)
        assert err < 1e-10, (name, key, err)
    with capsys.disabled():
        print("\nclass coverage (grid / discretization: [(cfg, a_global, nodes)], max rel err vs oracle):")
        for name, cls, err in rows:
            print(f"  {name:34s} {cls}  {err:.1e}")
    assert {c for c, _ in union} == set(range(NUM_SOLVER_CFGS)), sorted(union)
    assert {a for _, a in union} == {False, True}, sorted(union)
