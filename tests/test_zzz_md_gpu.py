"""GPU legs of the mixed-dimensional tests (tests/test_mdflow.py, tests/test_mdgrid.py): the coupled Jacobian of a whole
fracture network assembled by the device AD chain, against the reference's Jacobian / right-hand side / solution
(tests/golden/mdflow_*.npz) and against the block-by-block host restatement.  Named to run last."""
import numpy as np
import pytest

from test_mdflow import CASES, _check
from test_mdgrid import network, problem
from mdflow_io import load_mdflow


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_md_jacobian_gpu(name):
    import torch
    prob, Jref, bref, xref = load_mdflow(name)
    prob.discretize()
    Jh, bh = prob.assemble_host()
    for assemble in (prob.assemble_ad, prob.assemble):
        J, rhs = assemble()
        _check(J.to_scipy(), rhs.cpu().numpy(), Jref, bref, xref)
        assert abs(J.to_scipy() - Jh).max() <= 1e-12 * abs(Jh).max()
        _, r = assemble(torch.as_tensor(xref, device="cuda"))
        assert float(r.abs().max()) <= 1e-9 * np.abs(bref).max()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["hex", "tet"])
def test_md_problem_on_synthetic_network_gpu(kind):
    prob = problem(network(kind, n=6)[2], value=lambda x: 1.0 + x[1] - 2.0 * x[2])
    prob.discretize()
    Jh, bh = prob.assemble_host()
    for assemble in (prob.assemble_ad, prob.assemble):
        J, rhs = assemble()
        assert abs(J.to_scipy() - Jh).max() <= 1e-12 * abs(Jh).max()
        assert np.abs(rhs.cpu().numpy() - bh).max() <= 1e-12 * np.abs(bh).max()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["hex", "tet"])
def test_md_solve_on_device(kind):
    """``MixedDimensionalFlow.solve`` (BiCGStab on the pressure Schur complement, device SpMVs) against a direct solve
    of the coupled system."""
    import scipy.sparse.linalg as spla
    prob = problem(network(kind, n=8)[2], a=1e-3, kn=1.0, value=lambda x: 1.0 + x[0])
    prob.discretize()
    x, info = prob.solve(tol=1e-11)
    assert info["converged"] and info["true_relres"] < 1e-9, info
    J, rhs = prob.assemble()
    xh = spla.spsolve(J.to_scipy().tocsc(), rhs.cpu().numpy())
    assert np.linalg.norm(x.cpu().numpy() - xh) <= 1e-7 * np.linalg.norm(xh)


# ---- compressible flow: the reference's Newton loop on the device AD chain (tests/test_mdflow_nonlinear.py); kept last
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mdflownl_one_fracture", "mdflownl_three_fractures"])
def test_compressible_md_newton_gpu(name):
    from mdflow_io import load_mdflow_nonlinear
    from test_mdflow_nonlinear import check_linearization, check_time_step
    prob, d = load_mdflow_nonlinear(name)
    prob.discretize()
    check_linearization(prob, d, lambda t: t.cpu().numpy())
    check_time_step(prob, d, lambda t: t.cpu().numpy())


@pytest.mark.gpu
def test_poromechanics_model_gpu():
    """``pp.Poromechanics`` on the device AD chain, Newton updates by the fused Jacobi-BiCGStab (tests/test_poromech_model.py)."""
    from test_poromech_model import check, load_problem
    prob, d = load_problem()
    prob.discretize()
    hist = check(prob, d, lambda t: t.cpu().numpy())
    assert all(h.get("linear_converged", True) for h in hist), hist


@pytest.mark.gpu
def test_thermoporomechanics_model_gpu():
    """``pp.Thermoporomechanics`` on the device AD chain, Newton updates by the fused Jacobi-BiCGStab (tests/test_thm_model.py)."""
    from test_thm_model import check, load_problem
    prob, d = load_problem()
    prob.discretize()
    hist = check(prob, d, lambda t: t.cpu().numpy())
    assert all(h.get("linear_converged", True) for h in hist), hist


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mdthermal_one_fracture", "mdthermal_three_fractures"])
def test_mass_and_energy_balance_on_a_network_gpu(name):
    """``pp.MassAndEnergyBalance`` on a fracture network (tests/test_mdthermal.py) with the device sparse algebra."""
    from mdflow_io import load_mdthermal
    from test_mdthermal import check
    prob, d = load_mdthermal(name)
    prob.discretize()
    check(prob, d, lambda t: t.cpu().numpy())


@pytest.mark.gpu
def test_ad_functions_gpu():
    """``porepy_b200.ad_functions`` on the device against the reference's ``pp.ad.functions`` (tests/golden/ad_functions.npz)."""
    import torch
    from porepy_b200 import ad, ad_functions
    from porepy_b200.sparse import DeviceCsr
    from test_ad_functions import run_checks

    def make(v, j):
        return ad.DeviceAdArray(torch.as_tensor(v.copy(), device="cuda"), DeviceCsr(j))

    def to_host(g):
        if isinstance(g, ad.DeviceAdArray):
            return g.val.cpu().numpy(), g.jac.to_scipy()
        return g.cpu().numpy(), None
    run_checks(make, ad_functions, to_host)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["contact_model", "contact_sticking", "contact_open", "contact_mixed"])
def test_frictional_contact_gpu(name):
    """``pp.MomentumBalance`` with a sliding fracture on the device AD chain (tests/test_contact_model.py); the Newton
    updates of this saddle-point system are solved on the host in the test."""
    import torch
    from test_contact_model import check, load_problem
    prob, d = load_problem(name)
    prob.discretize()
    check(prob, d, lambda t: t.cpu().numpy(), lambda a: torch.as_tensor(np.asarray(a, float), device="cuda"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["contact_poromech", "contact_poromech_mixed"])
def test_fractured_poromechanics_with_contact_gpu(name):
    """``pp.Poromechanics`` on a fractured medium with frictional contact (tests/test_contact_poromech.py) on the device AD
    chain; the Newton updates of the saddle-point system are solved on the host in the test."""
    import torch
    from test_contact_poromech import check, load_problem
    prob, d = load_problem(name)
    prob.discretize()
    check(prob, d, lambda t: t.cpu().numpy(), lambda a: torch.as_tensor(np.asarray(a, float), device="cuda"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["contact_thm", "contact_thm_mixed"])
def test_fractured_thermoporomechanics_with_contact_gpu(name):
    """BASELINE config[4] as the reference states it: ``pp.Thermoporomechanics`` on a fractured medium with frictional
    contact (tests/test_contact_thm.py) on the device AD chain; Newton updates solved on the host in the test."""
    import torch
    from test_contact_thm import check, load_problem
    prob, d = load_problem(name)
    prob.discretize()
    check(prob, d, lambda t: t.cpu().numpy(), lambda a: torch.as_tensor(np.asarray(a, float), device="cuda"))
