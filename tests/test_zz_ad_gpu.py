"""Device-side forward-mode AD chain (porepy_b200/ad.py, csrc/sparse_ops.cu): SpGEMM / sparse add / diagonal scaling /
block concatenation against scipy, ``DeviceAdArray`` against the reference's own ``AdArray`` (stored results), and a
coupled Biot system assembled on the device from the device-resident outputs of ``discretize`` against the host
assembly (Jacobian entrywise, right-hand side, Newton update)."""
import os

import numpy as np
import pytest
import scipy.sparse as sps
import scipy.sparse.linalg as spla

import porepy_b200 as pb
from porepy_b200 import ad
from porepy_b200.sparse import DeviceCsr, LazyCsr

pytestmark = pytest.mark.gpu


def _rand(m, n, density, seed):
    a = sps.random(m, n, density, format="csr", random_state=seed, data_rvs=np.random.default_rng(seed).standard_normal)
    a.sort_indices()
    return a


def _close(ref, got, tol=1e-13):
    ref = sps.csr_matrix(ref)
    got = sps.csr_matrix(got)
    assert ref.shape == got.shape
    scale = max(abs(ref).max() if ref.nnz else 0.0, 1e-300)
    d = abs(ref - got)
    return (d.max() if d.nnz else 0.0) <= tol * scale


def test_sparse_kernels_match_scipy():
    A, B, A2 = _rand(300, 200, 0.05, 1), _rand(200, 250, 0.08, 2), _rand(300, 200, 0.03, 3)
    dA, dB, dA2 = DeviceCsr(A), DeviceCsr(B), DeviceCsr(A2)
    C = dA.matmul(dB).to_scipy()
    assert _close(A @ B, C) and C.has_sorted_indices and np.all(np.diff(C.indptr) >= 0)
    for r in range(C.shape[0]):                       # canonical rows: strictly increasing columns
        cols = C.indices[C.indptr[r]:C.indptr[r + 1]]
        assert np.all(np.diff(cols) > 0)
    assert _close(2.0 * A - 0.5 * A2, dA.axpby(2.0, dA2, -0.5).to_scipy())
    import torch
    d = torch.as_tensor(np.random.default_rng(4).standard_normal(300), device="cuda")
    e = torch.as_tensor(np.random.default_rng(5).standard_normal(200), device="cuda")
    assert _close(sps.diags(d.cpu().numpy()) @ A, dA.scaled(d).to_scipy())
    assert _close(A @ sps.diags(e.cpu().numpy()), dA.scaled(e, by_cols=True).to_scipy())
    Z = _rand(250, 200, 0.02, 6)
    ref = sps.bmat([[A, None], [Z @ sps.identity(200), B.T.tocsr() @ sps.identity(200)[:200, :250].T]], format="csr") \
        if False else sps.bmat([[A, A @ B], [None, Z @ B]], format="csr")
    got = DeviceCsr.bmat([[dA, dA.matmul(dB)], [None, DeviceCsr(Z).matmul(dB)]]).to_scipy()
    assert _close(ref, got)
    assert _close(sps.block_diag([A, B, A2], format="csr"), DeviceCsr.block_diag([dA, dB, dA2]).to_scipy())
    assert _close(sps.vstack([A, A2]), DeviceCsr.vstack([dA, dA2]).to_scipy())
    x = torch.as_tensor(np.random.default_rng(7).standard_normal(200), device="cuda")
    assert np.allclose((dA @ x).cpu().numpy(), A @ x.cpu().numpy(), rtol=1e-13, atol=1e-13)
    # a product whose rows collide heavily in the hash table (dense-ish)
    D1, D2 = _rand(64, 64, 0.6, 8), _rand(64, 64, 0.6, 9)
    assert _close(D1 @ D2, DeviceCsr(D1).matmul(DeviceCsr(D2)).to_scipy())


GOLDEN_ADARRAY = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ad_adarray.npz")


def adarray_case():
    """Two variables, the operators and the weights of the expression of
    ``test_device_adarray_matches_the_reference_adarray``."""
    rng = np.random.default_rng(0)
    n1, n2 = 40, 25
    v1, v2 = rng.standard_normal(n1), rng.standard_normal(n2)
    M = _rand(30, n1, 0.2, 11)
    N = _rand(30, n2, 0.3, 12)
    w = rng.standard_normal(30)
    return v1, v2, M, N, w


def test_device_adarray_matches_the_reference_adarray():
    """The expression evaluated by the reference's own ``AdArray`` is stored in tests/golden/ad_adarray.npz
    (tools/make_ad_functions_golden.py)."""
    v1, v2, M, N, w = adarray_case()
    x1, x2 = ad.variables([v1, v2])
    expr = (M @ x1) * (N @ x2) + 3.0 * (M @ x1) - (N @ x2) * w + 2.5
    expr = -expr + (M @ x1) * (M @ x1)
    d = np.load(GOLDEN_ADARRAY)
    ref_jac = sps.csr_matrix((d["jac__data"], d["jac__indices"], d["jac__indptr"]), shape=tuple(d["jac__shape"]))
    val, jac = expr.host()
    assert np.allclose(val, d["val"], rtol=1e-13, atol=1e-13)
    assert _close(ref_jac, jac)


def test_biot_system_assembled_on_the_device():
    """Two-field Biot step (the block system of the reference's test_biot.py) built by the device AD chain from the
    device-resident outputs of ``pb.Mpfa`` / ``pb.Biot``: nothing but the final comparison crosses PCIe."""
    g = pb.cart_grid_3d([6, 5, 4], perturb=0.2, seed=3)
    rng = np.random.default_rng(1)
    nc, nf = g.num_cells, g.num_faces
    k = pb.SecondOrderTensor(1 + rng.random(nc), 1 + rng.random(nc), 1 + rng.random(nc),
                             0.3 * rng.random(nc), 0.3 * rng.random(nc), 0.3 * rng.random(nc))
    bfc = g.get_all_boundary_faces()
    bc = pb.BoundaryCondition(g, bfc[g.face_centers[0, bfc] < 1e-10], "dir")
    C = pb.FourthOrderTensor(np.exp(0.3 * rng.standard_normal(nc)), np.exp(0.3 * rng.standard_normal(nc)))
    vbc = pb.BoundaryConditionVectorial(g, bfc[g.face_centers[2, bfc] < 1e-10], "dir")
    dflow = pb.initialize_data({}, "flow", {"second_order_tensor": k, "bc": bc})
    dmech = pb.initialize_data({}, "mech", {"fourth_order_tensor": C, "bc": vbc, "scalar_vector_mappings": {"flow": 0.8}})
    pb.Mpfa("flow").discretize(g, dflow)
    pb.Biot("mech").discretize(g, dmech)
    F, Mm = dflow[pb.DISCRETIZATION_MATRICES]["flow"], dmech[pb.DISCRETIZATION_MATRICES]["mech"]
    before = dict(LazyCsr.downloads)
    div, div3 = g.divergence(1), g.divergence(3)
    dt, storage = 0.1, 1e-2 * np.asarray(g.cell_volumes)
    u0, p0 = rng.standard_normal(3 * nc), rng.standard_normal(nc)
    ubc, pbc = 1e-2 * rng.standard_normal(3 * nf), rng.standard_normal(nf)
    u_prev, p_prev = rng.standard_normal(3 * nc), rng.standard_normal(nc)
    u, p = ad.variables([u0, p0])
    stress = ad.merged([Mm["stress"]]) @ u + ad.merged([Mm["scalar_gradient"]["flow"]]) @ p \
        + ad.as_device_csr(Mm["bound_stress"]) @ ad.device_vector(ubc)
    momentum = div3 @ stress
    flux = ad.merged([F["flux"]]) @ p + ad.as_device_csr(F["bound_flux"]) @ ad.device_vector(pbc)
    du = u - u_prev
    mass = ad.merged([Mm["displacement_divergence"]["flow"]]) @ du \
        + ad.merged([Mm["mpsa_consistency"]["flow"]]) @ (p - p_prev) + (p - p_prev) * storage + (div @ flux) * dt
    J, rhs = ad.assemble([momentum, mass])
    assert LazyCsr.downloads == before, "the device chain must not download the discretization matrices"
    # host assembly from downloaded copies of the same matrices
    S, G, BS = (sps.csr_matrix(Mm[k_]) if not isinstance(Mm[k_], dict) else sps.csr_matrix(Mm[k_]["flow"])
                for k_ in ("stress", "scalar_gradient", "bound_stress"))
    DD, CONS = sps.csr_matrix(Mm["displacement_divergence"]["flow"]), sps.csr_matrix(Mm["mpsa_consistency"]["flow"])
    FL, BF = sps.csr_matrix(F["flux"]), sps.csr_matrix(F["bound_flux"])
    J_ref = sps.bmat([[div3 @ S, div3 @ G], [DD, CONS + sps.diags(storage) + dt * (div @ FL)]], format="csr")
    r_mom = div3 @ (S @ u0 + G @ p0 + BS @ ubc)
    r_mass = DD @ (u0 - u_prev) + CONS @ (p0 - p_prev) + storage * (p0 - p_prev) + dt * (div @ (FL @ p0 + BF @ pbc))
    rhs_ref = -np.r_[r_mom, r_mass]
    assert _close(J_ref, J.to_scipy(), tol=1e-12)
    assert np.abs(rhs.cpu().numpy() - rhs_ref).max() <= 1e-11 * np.abs(rhs_ref).max()
    dx = spla.spsolve(sps.csc_matrix(J.to_scipy()), rhs.cpu().numpy())
    dx_ref = spla.spsolve(sps.csc_matrix(J_ref), rhs_ref)
    assert np.linalg.norm(dx - dx_ref) <= 1e-9 * np.linalg.norm(dx_ref)
