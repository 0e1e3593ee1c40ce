"""Thermo-poromechanics of a fractured medium with frictional contact -- BASELINE config[4] ("thermo-poromechanics +
frictional contact, fracture network, full Newton loop") as the reference states it: ``pp.Thermoporomechanics`` on a matrix
cut by fractures, every term and its Jacobian by ``DeviceAdArray`` on device-resident matrices.

The union of ``porepy_b200.fractured_poromech`` (poromechanics, fracture flow with jump-dependent aperture, contact),
``porepy_b200.thermoporomech`` (thermal stress, thermally expanding fluid, thermo-poromechanical porosity, internal energy)
and ``porepy_b200.mdthermal`` (Fourier and enthalpy fluxes on subdomains and interfaces), with the aperture in the
fracture's internal energy and in the interface Fourier law:

* fracture energy        vol a (rho c_f (T - T0) - p)        (porosity 1, specific volume a)
* interface Fourier law  eta - vol kappa_T (2 Pi (1 / a)) (Pi tr T - Pi T_f)                constitutive_laws.py:2342-2386
* fracture conductivity  k_f a: the fracture's Fourier flux is re-discretized with the iterate's aperture like its Darcy
                         flux (measured on the reference: both flux matrices x 1.002 at the second iterate); the matrix's
                         flux matrices stay those of the initial state.

Unknowns: [p matrix | p fractures | T matrix | T fractures | u | contact tractions | lambda | eta | eps | u_j]; equations:
[mass matrix | mass fractures | energy matrix | energy fractures | momentum | Darcy laws | Fourier laws | enthalpy laws |
force balances | normal laws | tangential laws].  ``contact.device_linear_solver`` solves the Newton steps on the device
(GMRES with the local blocks of ``block_layout``).  ``tests/golden/contact_thm*.npz`` pin the Jacobian at the zero state and at
the fourth Newton iterate, the residual history of the semismooth Newton loop and the converged state.
"""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np

from . import ad, ad_functions as fn
from .contact import local_block_layout, mortar_pairs, offsets_of
from .fractured_poromech import FracturedPoromechanics
from .fv import Mpfa, Upwind, UpwindCoupling
from .params import DISCRETIZATION_MATRICES, PARAMETERS, SecondOrderTensor


class FracturedThermoporomechanics(FracturedPoromechanics):
    """As ``FracturedPoromechanics``, plus: ``data[parameters][fourier_keyword]`` (``bc``) for the matrix and for every
    fracture (``FractureCoupling.data``); ``scalar_vector_mappings`` of the mechanics parameters hold the thermal-stress
    tensor under ``thermal_keyword``; ``fluid`` adds ``thermal_expansion, heat_capacity, conductivity,
    reference_temperature``; ``solid`` adds ``biot_coefficient, thermal_expansion, heat_capacity, conductivity, density``;
    ``bc`` adds the face arrays ``fourier``, ``enthalpy_flux`` and the object ``enthalpy_flux_type``;
    ``normal_thermal_conductivity``: one array per fracture interface."""

    enthalpy_upwind_keyword = "enthalpy_upwind"

    def __init__(self, sd, data: dict, fractures, fluid: dict, solid: dict, contact: dict, bc: dict,
                 normal_thermal_conductivity, flow_keyword: str = "flow", fourier_keyword: str = "fourier",
                 mechanics_keyword: str = "mechanics", thermal_keyword: str = "thermal"):
        super().__init__(sd, data, fractures, fluid, solid, contact, bc, flow_keyword, mechanics_keyword)
        self.tk, self.ck = fourier_keyword, thermal_keyword
        self.kappa_t = [np.asarray(v, float) for v in normal_thermal_conductivity]
        nfc = [f.num_cells for f in self.fractures]
        nm = [f.num_mortar for f in self.fractures]
        self.sizes = [self.nc] + nfc + [self.nc] + nfc + [3 * self.nc] + [3 * n for n in nfc] + nm + nm + nm + [3 * n for n in nm]
        self.offsets = np.concatenate(([0], np.cumsum(self.sizes))).astype(np.int64)

    def block_layout(self):
        """Local blocks of the Jacobian: p, T and u of every matrix cell (5, with the mass, energy and momentum
        balances), and per fracture cell its traction, pressure and temperature with lambda, eta, eps and u_j of its two
        mortar cells (17, with the fracture mass and energy balances, the contact laws and the Darcy, Fourier and
        enthalpy laws and force balances of the two mortar cells)."""
        nfr, o = len(self.fractures), self.offsets
        nfc = [f.num_cells for f in self.fractures]
        nm = [f.num_mortar for f in self.fractures]
        e = offsets_of([self.nc] + nfc + [self.nc] + nfc + [3 * self.nc] + nm + nm + nm + [3 * n for n in nm] + nfc
                       + [2 * n for n in nfc])
        return local_block_layout(
            self.nc, [mortar_pairs(f.p["mortar_to_secondary_avg"]) for f in self.fractures],
            [(o[0], 1), (o[1 + nfr], 1), (o[2 + 2 * nfr], 3)], [(e[0], 1), (e[1 + nfr], 1), (e[2 + 2 * nfr], 3)],
            [[(o[3 + 2 * nfr + j], 3, "fracture"), (o[1 + j], 1, "fracture"), (o[2 + nfr + j], 1, "fracture")]
             + [(o[3 + q * nfr + j], 1, "mortar") for q in (3, 4, 5)] + [(o[3 + 6 * nfr + j], 3, "mortar")]
             for j in range(nfr)],
            [[(e[3 + 6 * nfr + j], 1, "fracture"), (e[3 + 7 * nfr + j], 2, "fracture"), (e[1 + j], 1, "fracture"),
              (e[2 + nfr + j], 1, "fracture")] + [(e[3 + q * nfr + j], 1, "mortar") for q in (2, 3, 4)]
             + [(e[3 + 5 * nfr + j], 3, "mortar")] for j in range(nfr)])

    # ---- discretizations
    def _matrix_conductivity(self):
        phi = self.so.reference_porosity
        return np.full(self.nc, phi * self.fl.conductivity + (1.0 - phi) * self.so.conductivity)

    def _discretize_fracture(self, fc, aperture) -> None:
        super()._discretize_fracture(fc, aperture)
        fc.data.setdefault(PARAMETERS, {}).setdefault(self.tk, {})["second_order_tensor"] = SecondOrderTensor(
            self.fl.conductivity * np.asarray(aperture, float))          # porosity 1 in the fracture, specific volume a
        fc.data[PARAMETERS][self.tk].setdefault("ambient_dimension", 3)
        Mpfa(self.tk).discretize(fc.sd, fc.data)

    def discretize(self) -> None:
        self.data[PARAMETERS][self.tk]["second_order_tensor"] = SecondOrderTensor(self._matrix_conductivity())
        Mpfa(self.tk).discretize(self.sd, self.data)
        super().discretize()

    def _operands(self):
        fresh = self._const is None
        k = super()._operands()
        if fresh:
            csr, dev = ad.as_device_csr, ad.device_vector
            Fo = self.data[DISCRETIZATION_MATRICES][self.tk]
            M = self.data[DISCRETIZATION_MATRICES][self.mk]
            k.Fo = {key: csr(Fo[key]) for key in ("flux", "bound_flux", "bound_pressure_cell", "bound_pressure_face")}
            k.grad_t = csr(M["scalar_gradient"][self.ck])
            k.bct, k.bce = dev(self.bc["fourier"]), dev(self.bc["enthalpy_flux"])
            for j, fc in enumerate(self.fractures):
                k.fr[j].coef_t = dev(fc.volumes * self.kappa_t[j] * 2.0)
        return k

    # ---- constitutive laws
    def _density(self, p, t=None):
        fl = self.fl
        e = (p - fl.reference_pressure) * fl.compressibility
        if t is not None:
            e = e - (t - fl.reference_temperature) * fl.thermal_expansion
        return e.exp() * fl.density

    def _porosity(self, p, t, u, uj, k):
        so = self.so
        return super()._porosity(p, u, uj, k) \
            - (t - self.fl.reference_temperature) * ((so.biot_coefficient - so.reference_porosity) * so.thermal_expansion)

    def _group(self, parts):
        n = len(self.fractures)
        i = 0
        out = []
        for size in (1, n, 1, n, 1, n, n, n, n, n):
            out.append(parts[i:i + size])
            i += size
        p3, pf, t3, tf, u, t, lam, eta, eps, uj = out
        return p3[0], pf, t3[0], tf, u[0], t, lam, eta, eps, uj

    def update_discretizations(self, x) -> None:
        x = ad.device_vector(x)
        k = self._operands()
        p3, pf, _, _, _, _, lam, _, _, uj = self._parts(x)
        for j, fc in enumerate(self.fractures):
            self._discretize_fracture(fc, self._aperture(uj[j], k.fr[j]).cpu().numpy())
        b = k.bcq
        for j in range(len(self.fractures)):
            b = (k.fr[j].m2p @ lam[j]) + b
        q3 = ((k.F["flux"] @ p3) + (k.F["bound_flux"] @ b)).cpu().numpy()
        for kw, bc in ((self.mobility_keyword, self.bc["fluid_flux_type"]),
                       (self.enthalpy_upwind_keyword, self.bc["enthalpy_flux_type"])):
            prm = self.data.setdefault(PARAMETERS, {}).setdefault(kw, {})
            prm["darcy_flux"], prm["bc"] = q3, bc
            Upwind(kw).discretize(self.sd, self.data)
        for j, fc in enumerate(self.fractures):
            qf = self._fracture_flux(fc, k.fr[j], pf[j]).cpu().numpy()
            for kw, key in ((self.mobility_keyword, "fluid_flux_type"), (self.enthalpy_upwind_keyword, "enthalpy_flux_type")):
                prm = fc.data.setdefault(PARAMETERS, {}).setdefault(kw, {})
                prm["darcy_flux"] = qf
                prm["bc"] = fc.data[PARAMETERS][self.fk]["bc"] if fc.bc is None else fc.bc[key]
                Upwind(kw).discretize(fc.sd, fc.data)
            d = self._intf_data[j]
            d.setdefault(PARAMETERS, {}).setdefault(self.mobility_keyword, {})["darcy_flux"] = lam[j].cpu().numpy()
            UpwindCoupling(self.mobility_keyword).discretize(self.sd, fc.sd, SimpleNamespace(num_cells=fc.num_mortar),
                                                             self.data, fc.data, d)

    def equations(self, x, x_prev, dt: float) -> list:
        k, ct, fl, so = self._operands(), self.ct, self.fl, self.so
        csr = ad.as_device_csr
        nfr = len(self.fractures)
        mk, ek = self.mobility_keyword, self.enthalpy_upwind_keyword
        x, x_prev = ad.device_vector(x), ad.device_vector(x_prev)
        var = ad.variables([x[self.offsets[q]:self.offsets[q + 1]] for q in range(len(self.sizes))])
        p3, pf, t3, tf, u, t, lam, eta, eps, uj = self._group(var)
        p3n, pfn, t3n, tfn, un, _, _, _, _, ujn = self._parts(x_prev)
        t0 = fl.reference_temperature

        def weights(p, tt):
            w = self._density(p, tt) * (1.0 / fl.viscosity)
            return w, w * (tt - t0) * fl.heat_capacity
        w3, we3 = weights(p3, t3)
        wf, wef = zip(*[weights(pf[j], tf[j]) for j in range(nfr)]) if nfr else ((), ())
        ifl, enthalpy, b_flow, b_heat, b_mech = [], [], k.bcq, k.bct, k.ubc
        for j in range(nfr):
            q = k.fr[j]
            U = self._intf_data[j][DISCRETIZATION_MATRICES][mk]
            up, us = csr(U["upwind_primary"]), csr(U["upwind_secondary"])

            def upwinded(a3, af):
                return (up @ (q.p2m @ (k.trace @ a3))) + (us @ (q.s2m @ af))
            ifl.append(lam[j] * upwinded(w3, wf[j]))
            enthalpy.append(eps[j] - lam[j] * upwinded(we3, wef[j]))
            b_flow = (q.m2p @ lam[j]) + b_flow
            b_heat = (q.m2p @ eta[j]) + b_heat
            b_mech = (q.m2p3 @ uj[j]) + b_mech
        # ---- matrix
        Tm, Te = self.data[DISCRETIZATION_MATRICES][mk], self.data[DISCRETIZATION_MATRICES][ek]
        q3 = (k.F["flux"] @ p3) + (k.F["bound_flux"] @ b_flow)
        neu_m, neu_e = k.bcw, k.bce
        for j in range(nfr):
            neu_m = (k.fr[j].m2p @ ifl[j]) + neu_m
            neu_e = (k.fr[j].m2p @ eps[j]) + neu_e
        ff3 = q3 * (csr(Tm["transport"]) @ w3) + (csr(Tm["rhs_dir"]) @ (q3 * k.bcw)) + (csr(Tm["rhs_neu"]) @ neu_m)
        fe3 = q3 * (csr(Te["transport"]) @ we3) + (csr(Te["rhs_dir"]) @ (q3 * k.bce)) + (csr(Te["rhs_neu"]) @ neu_e)
        fo3 = (k.Fo["flux"] @ t3) + (k.Fo["bound_flux"] @ b_heat)
        phi, phi_n = self._porosity(p3, t3, u, uj, k), self._porosity(p3n, t3n, un, ujn, k)
        rho3, rho3n = self._density(p3, t3), self._density(p3n, t3n)
        mass3 = (rho3 * phi - rho3n * phi_n) * (k.vol * (1.0 / dt)) + (k.div @ ff3)

        def energy(p, tt, rho, por):
            dtm = tt - t0
            return (rho * dtm * fl.heat_capacity - p) * por + (dtm * (so.density * so.heat_capacity)) * (-por + 1.0)
        energy3 = (energy(p3, t3, rho3, phi) - energy(p3n, t3n, rho3n, phi_n)) * (k.vol * (1.0 / dt)) + (k.div @ (fe3 + fo3))
        stress = (k.stress @ u) + (k.bound @ b_mech) + (k.grad_p @ (p3 - fl.reference_pressure)) + (k.grad_t @ (t3 - t0))
        momentum = -(k.div3 @ stress)
        trace_p = (k.F["bound_pressure_cell"] @ p3) + (k.F["bound_pressure_face"] @ b_flow)
        trace_t = (k.Fo["bound_pressure_cell"] @ t3) + (k.Fo["bound_pressure_face"] @ b_heat)
        mass_f, energy_f, darcy, fourier, force, normal, tangential = [], [], [], [], [], [], []
        for j, fc in enumerate(self.fractures):
            q = k.fr[j]
            a, a_n = self._aperture(uj[j], q), self._aperture(ujn[j], q)
            Tf, Tef = fc.data[DISCRETIZATION_MATRICES][mk], fc.data[DISCRETIZATION_MATRICES][ek]
            qf = self._fracture_flux(fc, q, pf[j])
            Fof = fc.data[DISCRETIZATION_MATRICES][self.tk]
            fof = csr(Fof["flux"]) @ tf[j]
            if q.bc is not None:
                fof = fof + (csr(Fof["bound_flux"]) @ q.bc["fourier"])
            rhof, rhofn = self._density(pf[j], tf[j]), self._density(pfn[j], tfn[j])
            mass_f.append((a * rhof - a_n * rhofn) * (q.vol * (1.0 / dt))
                          + (q.div @ self._advective(Tf, qf, wf[j], q, "fluid_flux")) - (q.m2s @ ifl[j]))
            ef = rhof * (tf[j] - t0) * fl.heat_capacity - pf[j]                  # porosity 1: no solid part
            efn = rhofn * (tfn[j] - t0) * fl.heat_capacity - pfn[j]
            energy_f.append((a * ef - a_n * efn) * (q.vol * (1.0 / dt))
                            + (q.div @ (self._advective(Tef, qf, wef[j], q, "enthalpy_flux") + fof))
                            - (q.m2s @ (eta[j] + eps[j])))
            inv_a = q.s2m @ a.reciprocal()
            darcy.append(lam[j] - ((q.p2m @ trace_p) - (q.s2m @ pf[j])) * inv_a * q.coef)
            fourier.append(eta[j] - ((q.p2m @ trace_t) - (q.s2m @ tf[j])) * inv_a * q.coef_t)
            force.append((q.p2m3 @ (stress * k.outward)) + (q.traction @ t[j]) + (q.pressure_load @ pf[j]))
            jump, jump_n = q.jump @ uj[j], q.jump @ ujn[j]
            t_n, u_n = q.sel_n @ t[j], q.sel_n @ jump
            t_t, u_t, u_t_prev = q.sel_t @ t[j], q.sel_t @ jump, q.sel_t @ jump_n
            gap = fn.l2_norm(2, u_t) * float(np.tan(ct.dilation_angle)) + ct.reference_gap
            normal.append(t_n + fn.maximum(-t_n - (u_n - gap) * ct.numerical_constant, 0.0))
            s = t_t + (u_t - u_t_prev) * ct.numerical_constant
            b_p = fn.maximum(t_n * (-ct.friction_coefficient), 0.0)
            chi = q.s2t @ fn.characteristic_function(ct.open_state_tolerance, b_p).val
            tangential.append(((q.s2t @ b_p) * s - (q.s2t @ fn.maximum(b_p, fn.l2_norm(2, s))) * t_t) * (1.0 - chi)
                              + t_t * chi)
        return [mass3] + mass_f + [energy3] + energy_f + [momentum] + darcy + fourier + enthalpy + force + normal + tangential
