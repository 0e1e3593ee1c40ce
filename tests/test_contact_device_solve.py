"""The contact models' Newton steps solved on the device: the local-block layouts of ``FracturedMomentumBalance``,
``FracturedPoromechanics`` and ``FracturedThermoporomechanics``, restarted GMRES (``krylov.gmres``) with the local-block
inverse preconditioner (``krylov.LocalBlocks``), ``contact.device_linear_solver`` in the semismooth Newton loops of the
eight contact fixtures, and the sign / local-frame rule of ``mdgrid.fracture_contacts`` that generates contact problems
of any size.  CPU: eager GMRES with the NumPy twin of the block kernels (tests/local_blocks_np.py)."""
import numpy as np
import pytest
import scipy.sparse as sps
import scipy.sparse.linalg as spla

from porepy_b200 import krylov, mdgrid
from local_blocks_np import NumpyLocalBlocks, block_inverses
import test_contact_model as tcm
import test_contact_poromech as tcp
import test_contact_thm as tct

MODULES = {name: mod for mod in (tcm, tcp, tct) for name in mod.CASES}
FIXTURES = list(MODULES)
BLOCK_SIZES = {tcm: (3, 9), tcp: (4, 12), tct: (5, 17)}


def device_order_jacobian(name):
    """The fixture's ``iterate_jacobian`` / ``iterate_rhs`` in the model's row and column order."""
    mod = MODULES[name]
    prob, d = mod.load_problem(name)
    J = mod._csr(d, "iterate_jacobian")
    rm = d["row_map"] if "row_map" in d else np.arange(J.shape[0])
    cm = d["column_map"]
    return prob, d, sps.csr_matrix(J[rm][:, cm]), d["iterate_rhs"][rm]


class HostOperator:
    def __init__(self, a):
        self.a = sps.csr_matrix(a)

    def matvec(self, v):
        import torch
        return torch.as_tensor(self.a @ v.numpy())


def seeded_nonsymmetric(n=300, seed=3):
    """A well-posed nonsymmetric sparse matrix (diagonal shift + random couplings) and its layout of 1..6-wide blocks."""
    rng = np.random.default_rng(seed)
    a = sps.random(n, n, density=0.03, random_state=rng) - sps.random(n, n, density=0.03, random_state=rng)
    a = sps.csr_matrix(a + sps.diags(2.0 + rng.random(n)))
    sizes = []
    while sum(sizes) < n:
        sizes.append(min(int(rng.integers(1, 7)), n - sum(sizes)))
    from types import SimpleNamespace
    perm = rng.permutation(n).astype(np.int64)            # scattered blocks that hold their diagonal entries
    layout = SimpleNamespace(ptr=np.concatenate(([0], np.cumsum(sizes))).astype(np.int64), rows=perm, cols=perm.copy())
    return a, layout, rng.standard_normal(n)


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", FIXTURES)
def test_block_layout_is_a_bijection_with_the_expected_blocks(name):
    prob, d, J, _ = device_order_jacobian(name)
    L = prob.block_layout()
    krylov.check_block_layout(L, prob.num_dofs)
    sizes = np.diff(L.ptr)
    nc = prob.sd.num_cells
    nfc = sum(f.num_cells for f in prob.fractures)
    small, large = BLOCK_SIZES[MODULES[name]]
    assert np.array_equal(sizes, np.r_[np.full(nc, small), np.full(nfc, large)])
    inv = block_inverses(J, L)
    assert all(np.isfinite(m).all() for m in inv)


@pytest.mark.parametrize("name", FIXTURES)
def test_eager_gmres_matches_the_direct_solve(name):
    import torch
    prob, d, J, b = device_order_jacobian(name)
    P = NumpyLocalBlocks(prob.block_layout()).factor(J)
    x, info = krylov.gmres(HostOperator(J), torch.as_tensor(b), precond=P, tol=1e-12)
    ref = spla.spsolve(J.tocsc(), b)
    assert info["converged"] and info["relres"] <= 1e-12, info
    assert np.linalg.norm(x.numpy() - ref) <= 1e-10 * np.linalg.norm(ref), info


def test_eager_gmres_restarts():
    import torch
    a, layout, b = seeded_nonsymmetric()
    P = NumpyLocalBlocks(layout).factor(a)
    x, info = krylov.gmres(HostOperator(a), torch.as_tensor(b), precond=P, tol=1e-12, restart=7)
    ref = spla.spsolve(a.tocsc(), b)
    assert info["converged"] and info["restarts"] >= 1 and info["iterations"] > 7, info
    assert np.linalg.norm(x.numpy() - ref) <= 1e-10 * np.linalg.norm(ref), info
    x2, info2 = krylov.gmres(HostOperator(a), torch.as_tensor(b), tol=1e-12, restart=20)   # no preconditioner
    assert info2["converged"] and np.linalg.norm(x2.numpy() - ref) <= 1e-10 * np.linalg.norm(ref), info2


def test_eager_gmres_zero_rhs():
    import torch
    a, layout, _ = seeded_nonsymmetric()
    x, info = krylov.gmres(HostOperator(a), torch.zeros(a.shape[0], dtype=torch.float64),
                           precond=NumpyLocalBlocks(layout).factor(a))
    assert info["iterations"] == 0 and info["converged"] and not x.abs().max()


def test_singular_block_is_named():
    a, layout, _ = seeded_nonsymmetric()
    a = a.tolil()
    b = 5
    r = layout.rows[layout.ptr[b]:layout.ptr[b + 1]]
    c = layout.cols[layout.ptr[b]:layout.ptr[b + 1]]
    for i in r:
        a[i, c] = 0.0
    with pytest.raises(ValueError, match=r"Error in inversion of local linear systems \(block 5 "):
        block_inverses(a.tocsr(), layout)


def test_non_finite_block_is_named():
    a, layout, _ = seeded_nonsymmetric()
    b = 7
    r = layout.rows[layout.ptr[b]:layout.ptr[b + 1]]
    c = layout.cols[layout.ptr[b]:layout.ptr[b + 1]]
    a = a.tolil()
    a[r[-1], c[0]] = np.nan
    with pytest.raises(ValueError, match=r"Error in inversion of local linear systems \(block 7 "):
        block_inverses(a.tocsr(), layout)


def test_layout_checks():
    from types import SimpleNamespace
    with pytest.raises(ValueError, match="bijection"):
        krylov.check_block_layout(SimpleNamespace(ptr=np.array([0, 2, 3]), rows=np.array([0, 1, 1]),
                                                  cols=np.array([0, 1, 2])))
    with pytest.raises(ValueError, match="1..32"):
        krylov.check_block_layout(SimpleNamespace(ptr=np.array([0, 33]), rows=np.arange(33), cols=np.arange(33)))
    from porepy_b200.contact import mortar_pairs
    with pytest.raises(NotImplementedError):
        mortar_pairs(sps.csr_matrix(np.array([[1.0, 1.0, 1.0]])))


@pytest.mark.parametrize("name", FIXTURES)
def test_fracture_contact_rule_reproduces_the_fixture(name):
    mod = MODULES[name]
    prob, d = mod.load_problem(name)
    m2p = mod._csr(d, "mortar_to_primary_avg")
    sign = mdgrid.mortar_signs(prob.sd, m2p)
    assert np.array_equal(sign, d["mortar_sign"])
    L = mdgrid.fracture_local_coordinates(prob.sd, m2p, sign, int(d["mortar_to_secondary_avg__shape"][0]))
    assert abs(L - mod._csr(d, "local_coordinates")).max() <= 1e-14


def test_fracture_contacts_of_a_generated_network():
    import porepy_b200 as pb
    g = pb.cart_grid_3d([4, 4, 4])
    net = mdgrid.split_fractures(g, [mdgrid.faces_on_rectangle(g, 0, 0.5, (0.25, 0.25), (0.75, 0.75))])
    (fc,) = mdgrid.fracture_contacts(net)
    assert fc.num_cells == 4 and fc.num_mortar == 8
    sign = np.diag(fc.sign.toarray())[::3]
    assert sorted(np.unique(sign)) == [-1.0, 1.0] and sign.sum() == 0
    R = fc.rotation.toarray()[:3, :3]
    assert np.allclose(R @ R.T, np.eye(3)) and np.isclose(np.linalg.det(R), 1.0)
    # the normal points from the -1 side to the +1 side: here from x > 1/2 to x < 1/2
    cf = sps.csr_matrix(net.matrix.cell_faces)
    face = fc.m2p.tocsc()[:, 3 * int(np.flatnonzero(sign < 0)[0])].indices[0] // 3
    cell = cf[face].indices[0]
    assert np.sign(R[2, 0]) == -np.sign(net.matrix.cell_centers[0, cell] - 0.5)


# ---------------------------------------------------------------------------------------------------------------- GPU
def _cuda(a):
    import torch
    return torch.as_tensor(np.asarray(a, float), device="cuda")


@pytest.mark.gpu
def test_local_blocks_factor_matches_numpy():
    from porepy_b200.sparse import DeviceCsr
    for name in FIXTURES:
        prob, d, J, _ = device_order_jacobian(name)
        L = prob.block_layout()
        ref = block_inverses(J, L)
        lb = krylov.LocalBlocks(L).factor(DeviceCsr(J))
        got = lb.inv.cpu().numpy()
        flat = np.concatenate([m.ravel() for m in ref])
        assert np.abs(got - flat).max() <= 1e-12 * np.abs(flat).max(), name
        r = np.random.default_rng(1).standard_normal(J.shape[0])
        z = lb.apply(_cuda(r)).cpu().numpy()
        zr = NumpyLocalBlocks(L).factor(J).apply(__import__("torch").as_tensor(r)).numpy()
        assert np.abs(z - zr).max() <= 1e-12 * np.abs(zr).max(), name
    a, layout, _ = seeded_nonsymmetric()
    a = a.tolil()
    b = 5
    for i in layout.rows[layout.ptr[b]:layout.ptr[b + 1]]:
        a[i, layout.cols[layout.ptr[b]:layout.ptr[b + 1]]] = 0.0
    lb = krylov.LocalBlocks(layout)
    with pytest.raises(ValueError, match=r"Error in inversion of local linear systems \(block 5 "):
        lb.factor(DeviceCsr(a.tocsr()))


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["first", "last", "pivot"])
def test_local_blocks_factor_names_a_block_with_nan(entry):
    """A NaN anywhere in a block (e.g. from a diverging Newton step) is reported for that block, never inverted."""
    from porepy_b200.sparse import DeviceCsr
    prob, d, J, _ = device_order_jacobian("contact_thm")
    L = prob.block_layout()
    nb = len(L.ptr) - 1
    for b in (3, nb - 2):                                        # a 5-wide matrix-cell block and a 17-wide fracture block
        r = L.rows[L.ptr[b]:L.ptr[b + 1]]
        c = L.cols[L.ptr[b]:L.ptr[b + 1]]
        Jb = J.tolil()
        i, j = {"first": (r[0], c[0]), "last": (r[-1], c[-1]), "pivot": (r[1], c[0])}[entry]
        Jb[i, j] = np.nan
        with pytest.raises(ValueError, match=rf"Error in inversion of local linear systems \(block {b} "):
            krylov.LocalBlocks(L).factor(DeviceCsr(Jb.tocsr()))
    # the layout's blocks are still factorised where the matrix is finite
    krylov.LocalBlocks(L).factor(DeviceCsr(J))


@pytest.mark.gpu
def test_device_gmres_refuses_a_foreign_preconditioner():
    from porepy_b200.sparse import DeviceCsr
    a, layout, b = seeded_nonsymmetric()
    with pytest.raises(TypeError, match="LocalBlocks"):
        krylov.gmres(DeviceCsr(a), _cuda(b), precond=NumpyLocalBlocks(layout).factor(a))


@pytest.mark.gpu
def test_device_gmres_matches_the_direct_solve():
    from porepy_b200.sparse import DeviceCsr
    report = []
    for name in FIXTURES:
        prob, d, J, b = device_order_jacobian(name)
        lb = krylov.LocalBlocks(prob.block_layout())
        Jd = DeviceCsr(J)
        lb.factor(Jd)
        x, info = krylov.gmres(Jd, _cuda(b), precond=lb, tol=1e-12)
        ref = spla.spsolve(J.tocsc(), b)
        assert info["converged"] and info["relres"] <= 1e-12, (name, info)
        assert np.linalg.norm(x.cpu().numpy() - ref) <= 1e-10 * np.linalg.norm(ref), (name, info)
        report.append((name, info["iterations"], info["restarts"], info["host_syncs"]))
    a, layout, b = seeded_nonsymmetric()
    ad = DeviceCsr(a)
    lb = krylov.LocalBlocks(layout).factor(ad)
    ref = spla.spsolve(a.tocsc(), b)
    x, info = krylov.gmres(ad, _cuda(b), precond=lb, tol=1e-12, restart=7)
    assert info["converged"] and info["restarts"] >= 1, info
    assert np.linalg.norm(x.cpu().numpy() - ref) <= 1e-10 * np.linalg.norm(ref), info
    x, info0 = krylov.gmres(ad, _cuda(b), tol=1e-12, restart=20)
    assert info0["converged"] and np.linalg.norm(x.cpu().numpy() - ref) <= 1e-10 * np.linalg.norm(ref), info0
    x, info_z = krylov.gmres(ad, _cuda(np.zeros_like(b)), precond=lb)
    assert info_z["iterations"] == 0 and info_z["converged"] and not x.abs().max()
    print("device GMRES (name, iterations, restarts, host syncs):", report, (info["iterations"], info["restarts"],
                                                                           info["host_syncs"]))


def _newton_acceptance(mod, prob, d, x, hist, nref):
    cm = d["column_map"]
    ref = d["residual_norms"]
    assert hist[-1]["residual"] <= 1e-10 * hist[0]["residual"] and len(hist) <= len(ref) + 1, hist
    for mine, theirs in zip(hist[:nref], ref[:nref]):
        if theirs > 1e-9 * ref[0]:
            assert abs(mine["residual"] - theirs) <= 0.05 * theirs, (hist, ref)
    xh = x.cpu().numpy()
    assert np.linalg.norm(xh - d["solution"][cm]) <= 1e-8 * np.linalg.norm(d["solution"])
    return xh


def _tractions(mod, prob, xh):
    nfr = len(prob.fractures)
    q = {tcm: 1, tcp: 2 + nfr, tct: 3 + 2 * nfr}[mod]
    return xh[prob.offsets[q]:prob.offsets[q + 1]].reshape(-1, 3)


@pytest.mark.gpu
@pytest.mark.parametrize("name", FIXTURES)
def test_newton_loop_with_the_device_solver(name, monkeypatch):
    from porepy_b200.contact import device_linear_solver
    from porepy_b200.sparse import DeviceCsr
    mod = MODULES[name]
    prob, d = mod.load_problem(name)
    prob.discretize()
    solver = device_linear_solver(prob)

    def no_download(self):
        raise AssertionError("a Jacobian left the device")
    monkeypatch.setattr(DeviceCsr, "to_scipy", no_download)
    cm = d["column_map"]
    if mod is tcm:
        x, hist = prob.time_step(d["previous"], solver, tol=1e-11)
    else:
        x, hist = prob.time_step(d["previous"][cm], float(d["dt"]), solver, tol=1e-11)
    monkeypatch.undo()
    assert len(solver.history) == len(hist) - 1 and all(i["converged"] for i in solver.history)
    xh = _newton_acceptance(mod, prob, d, x, hist, 4 if mod is tcm else 5)
    t = _tractions(mod, prob, xh)
    mu = float(d["friction_coefficient"])
    is_open = np.abs(t[:, 2]) < 1e-12
    assert np.all(np.abs(t[is_open]) < 1e-12) and np.all(t[~is_open, 2] < 0)
    assert np.all(np.linalg.norm(t[~is_open, :2], axis=1) <= mu * np.abs(t[~is_open, 2]) * (1 + 1e-8))
    print(name, [(i["iterations"], i["restarts"], i["host_syncs"]) for i in solver.history])


@pytest.mark.gpu
def test_generated_contact_problem_device_vs_direct():
    import torch
    from porepy_b200.contact import device_linear_solver
    from tools.contact_problem import generated_contact_problem
    prob, _ = generated_contact_problem(16, "hex", 1)
    prob.discretize()
    x0 = torch.zeros(prob.num_dofs, dtype=torch.float64, device="cuda")
    J, rhs = prob.linearize(x0, x0)
    solver = device_linear_solver(prob)
    dx = solver(J, rhs).cpu().numpy()
    ref = spla.spsolve(J.to_scipy().tocsc(), rhs.cpu().numpy())
    assert np.linalg.norm(dx - ref) <= 1e-8 * np.linalg.norm(ref), solver.history

    def direct(Jd, r):
        return _cuda(spla.spsolve(Jd.to_scipy().tocsc(), r.cpu().numpy()))
    xd, hd = prob.time_step(x0, direct, tol=1e-11)
    xg, hg = prob.time_step(x0, device_linear_solver(prob), tol=1e-11)
    assert len(hd) == len(hg), (hd, hg)
    for a, b in zip(hd, hg):
        if a["residual"] > 1e-9 * hd[0]["residual"]:
            assert abs(a["residual"] - b["residual"]) <= 1e-6 * a["residual"], (hd, hg)
    xd, xg = xd.cpu().numpy(), xg.cpu().numpy()
    assert np.linalg.norm(xg - xd) <= 1e-8 * np.linalg.norm(xd)
    print("generated 16^3 hex:", prob.num_dofs, "unknowns,", len(hg) - 1, "Newton steps,",
          [i["iterations"] for i in solver.history])
