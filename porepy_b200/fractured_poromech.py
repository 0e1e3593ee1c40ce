"""Poromechanics of a fractured medium with frictional contact -- the reference's ``pp.Poromechanics`` on a matrix cut by
fractures, BASELINE configs[3] + [4] in one model: Biot poromechanics in the 3-D matrix (``porepy_b200.Mpfa`` + ``Biot``),
compressible flow in the 2-D fractures whose aperture follows the displacement jump, the interface Darcy law with that
aperture, the fluid pressure acting on the fracture walls, and the semismooth contact laws -- every term and its Jacobian
by ``DeviceAdArray`` on device-resident matrices.

Couplings on top of ``porepy_b200.poromech`` (matrix), ``mdflow_nl`` (fracture flow, interface law) and ``contact``
(interface force balance, complementarity laws):

* aperture               a = max([u]_n + a_res, a_res)                       constitutive_laws.py:307-365
* fracture fluid mass    vol a rho(p_f)      (specific volume a, porosity 1)  constitutive_laws.py:203-282, 4509-4534
* interface Darcy law    lambda - vol kappa (2 Pi (1 / a)) (Pi tr p - Pi p_f): the normal gradient follows a
* matrix porosity        displacement_divergence u + boundary_displacement_divergence (u_b + Pi u_j)
* matrix stress          stress u + bound_stress (u_b + Pi u_j) + scalar_gradient (p - p0)
* force balance          ... + vol n_out Pi p_f         (``fracture_pressure_stress``, constitutive_laws.py:3470-3492)

As in the reference's Newton loop (``Poromechanics.add_nonlinear_darcy_flux_discretization``, models/poromechanics.py), the
fracture flux is RE-DISCRETIZED in front of every linearization with the tangential permeability times the current
aperture (``operator_to_SecondOrderTensor``: the specific volume of the iterate; not differentiated), next to the
upwinding.  Unknowns: [p matrix | p fractures | u | contact tractions | lambda | u_j]; equations:
[mass matrix | mass fractures | momentum | Darcy laws | force balances | normal laws | tangential laws] (the fixtures carry
the maps to the reference's numbering).  One matrix subdomain, fractures without intersections; saddle-point Jacobian:
``contact.device_linear_solver`` solves the Newton steps on the device (GMRES with the local blocks of ``block_layout``),
and ``time_step`` takes any ``linear_solver(J, rhs) -> dx``.  ``tests/golden/contact_poromech*.npz`` pin Jacobian, residual, the residual
history of the semismooth Newton loop and the converged state.
"""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np
import scipy.sparse as sps

from . import ad, ad_functions as fn
from .contact import local_block_layout, mortar_pairs, offsets_of
from .fv import Biot, Mpfa, Upwind, UpwindCoupling
from .params import DISCRETIZATION_MATRICES, PARAMETERS


class FractureCoupling:
    """One fracture: its grid and data dictionary (``parameters[flow_keyword]``: ``bc``, ``ambient_dimension``; the
    ``second_order_tensor`` entry is written at every linearization: ``intrinsic_permeability`` (3, 3, nfc) times the
    aperture), the eight scalar mortar projections of its two-sided interface (``*_int`` / ``*_avg`` of the
    reference's ``MortarGrid``), ``mortar_sign``, ``mortar_volumes``, ``local_coordinates`` (3 nfc x 3 nfc) and the normal
    permeability per mortar cell; ``bc``: boundary data of a fracture that reaches the domain boundary."""

    def __init__(self, sd, data, projections: dict, mortar_sign, mortar_volumes, local_coordinates, normal_permeability,
                 intrinsic_permeability, bc: dict | None = None):
        self.sd, self.data = sd, data
        # boundary data of a fracture that reaches the domain boundary: face arrays ``flow``, ``fluid_flux`` (and
        # ``fourier``, ``enthalpy_flux``) plus the objects ``fluid_flux_type`` (``enthalpy_flux_type``); None: closed tips
        self.bc = bc
        self.k_intrinsic = np.asarray(intrinsic_permeability, float)
        self.p = {k: sps.csr_matrix(v) for k, v in projections.items()}
        self.sign = np.asarray(mortar_sign, float)
        self.volumes = np.asarray(mortar_volumes, float)
        self.rotation = sps.csr_matrix(local_coordinates)
        self.kappa = np.asarray(normal_permeability, float)
        self.num_cells, self.num_mortar = int(sd.num_cells), int(self.sign.size)


class FracturedPoromechanics:
    """``sd`` / ``data``: the matrix grid (fracture faces split) with ``parameters[flow_keyword]`` and
    ``parameters[mechanics_keyword]`` (``scalar_vector_mappings`` = {flow_keyword: Biot coefficient}).  ``bc``: dict of face
    arrays ``flow``, ``mechanics`` (3 nf), ``fluid_flux`` and the object ``fluid_flux_type``.  ``fluid``: ``compressibility,
    density, viscosity, reference_pressure``; ``solid``: ``reference_porosity, n_inv, residual_aperture``; ``contact``: the
    constants of ``porepy_b200.contact``."""

    mobility_keyword = "mobility"

    def __init__(self, sd, data: dict, fractures, fluid: dict, solid: dict, contact: dict, bc: dict,
                 flow_keyword: str = "flow", mechanics_keyword: str = "mechanics"):
        if int(sd.dim) != 3:
            raise NotImplementedError("a 3-D matrix grid is expected")
        self.sd, self.data = sd, data
        self.fractures = list(fractures)
        self.fk, self.mk = flow_keyword, mechanics_keyword
        self.fl = SimpleNamespace(**{k: float(v) for k, v in fluid.items()})
        self.so = SimpleNamespace(**{k: float(v) for k, v in solid.items()})
        self.ct = SimpleNamespace(**{k: float(v) for k, v in contact.items()})
        self.bc = bc
        self.nc, self.nf = int(sd.num_cells), int(sd.num_faces)
        nfc = [f.num_cells for f in self.fractures]
        nm = [f.num_mortar for f in self.fractures]
        self.sizes = [self.nc] + nfc + [3 * self.nc] + [3 * n for n in nfc] + nm + [3 * n for n in nm]
        self.offsets = np.concatenate(([0], np.cumsum(self.sizes))).astype(np.int64)
        self._intf_data = [{} for _ in self.fractures]
        self._const = None

    @property
    def num_dofs(self) -> int:
        return int(self.offsets[-1])

    def block_layout(self):
        """Local blocks of the Jacobian: p and u of every matrix cell (4, with the mass and momentum balances), and per
        fracture cell its traction and pressure with lambda and u_j of its two mortar cells (12, with the fracture mass
        balance, the contact laws and the Darcy laws and force balances of the two mortar cells)."""
        nfr, o = len(self.fractures), self.offsets
        nfc = [f.num_cells for f in self.fractures]
        nm = [f.num_mortar for f in self.fractures]
        e = offsets_of([self.nc] + nfc + [3 * self.nc] + nm + [3 * n for n in nm] + nfc + [2 * n for n in nfc])
        return local_block_layout(
            self.nc, [mortar_pairs(f.p["mortar_to_secondary_avg"]) for f in self.fractures],
            [(o[0], 1), (o[1 + nfr], 3)], [(e[0], 1), (e[1 + nfr], 3)],
            [[(o[2 + nfr + j], 3, "fracture"), (o[1 + j], 1, "fracture"), (o[2 + 2 * nfr + j], 1, "mortar"),
              (o[2 + 3 * nfr + j], 3, "mortar")] for j in range(nfr)],
            [[(e[2 + 3 * nfr + j], 1, "fracture"), (e[2 + 4 * nfr + j], 2, "fracture"), (e[1 + j], 1, "fracture"),
              (e[2 + nfr + j], 1, "mortar"), (e[2 + 2 * nfr + j], 3, "mortar")] for j in range(nfr)])

    def _discretize_fracture(self, fc, aperture) -> None:
        from .params import SecondOrderTensor
        fc.data[PARAMETERS][self.fk]["second_order_tensor"] = SecondOrderTensor.from_values(
            fc.k_intrinsic * np.asarray(aperture, float)[None, None, :])
        Mpfa(self.fk).discretize(fc.sd, fc.data)

    def discretize(self) -> None:
        """Matrix: Darcy flux and the Biot terms (once).  Fractures: Darcy flux at the residual aperture (re-discretized
        by ``update_discretizations`` at every iterate)."""
        Mpfa(self.fk).discretize(self.sd, self.data)
        Biot(self.mk).discretize(self.sd, self.data)
        for f in self.fractures:
            self._discretize_fracture(f, np.full(f.num_cells, self.so.residual_aperture))
        self._const = None

    def _operands(self):
        if self._const is None:
            csr, dev = ad.as_device_csr, ad.device_vector
            i3 = sps.identity(3, format="csr")
            F = self.data[DISCRETIZATION_MATRICES][self.fk]
            M = self.data[DISCRETIZATION_MATRICES][self.mk]
            cf = sps.csr_matrix(self.sd.cell_faces)
            frac_faces = np.asarray(self.sd.tags["fracture_faces"], bool)
            out = np.where(frac_faces, np.asarray(cf.sum(axis=1)).ravel(), 0.0)
            vol = np.asarray(self.sd.cell_volumes, float)
            k = SimpleNamespace(
                div=csr(sps.csr_matrix(self.sd.cell_faces.T)), div3=csr(sps.kron(sps.csr_matrix(self.sd.cell_faces.T), i3).tocsr()),
                trace=csr(abs(cf)), vol=dev(vol), inv_vol=dev(1.0 / vol),
                F={key: csr(F[key]) for key in ("flux", "bound_flux", "bound_pressure_cell", "bound_pressure_face")},
                stress=csr(M["stress"]), bound=csr(M["bound_stress"]), grad_p=csr(M["scalar_gradient"][self.fk]),
                div_u=csr(M["displacement_divergence"][self.fk]), div_u_b=csr(M["boundary_displacement_divergence"][self.fk]),
                cons=csr(M["mpsa_consistency"][self.fk]), outward=dev(np.repeat(out, 3)),
                bcq=dev(self.bc["flow"]), ubc=dev(self.bc["mechanics"]), bcw=dev(self.bc["fluid_flux"]), fr=[])
            for fc in self.fractures:
                n, p = fc.num_cells, fc.p
                sel_n = sps.csr_matrix((np.ones(n), (np.arange(n), 3 * np.arange(n) + 2)), shape=(n, 3 * n))
                sel_t = sps.csr_matrix((np.ones(2 * n), (np.arange(2 * n), 3 * np.repeat(np.arange(n), 2)
                                                         + np.tile([0, 1], n))), shape=(2 * n, 3 * n))
                s2t = sps.csr_matrix((np.ones(2 * n), (np.arange(2 * n), np.repeat(np.arange(n), 2))), shape=(2 * n, n))
                sign3 = sps.diags(np.repeat(fc.sign, 3))
                jump = fc.rotation @ sps.kron(p["mortar_to_secondary_avg"], i3) @ sign3
                trac = sps.diags(np.repeat(fc.volumes, 3) * self.ct.characteristic_traction) @ sign3 \
                    @ sps.kron(p["secondary_to_mortar_int"], i3) @ fc.rotation.T
                # unit normal of the primary face of every mortar cell, pointing out of the matrix, times the mortar volume
                pf = p["primary_to_mortar_avg"].tocsr().indices
                n_out = np.asarray(self.sd.face_normals)[:, pf] / np.asarray(self.sd.face_areas)[pf] * out[pf]
                rows = np.arange(3 * fc.num_mortar)
                pressure_load = sps.csr_matrix(((n_out * fc.volumes).ravel("F"), (rows, np.repeat(np.arange(fc.num_mortar), 3))),
                                               shape=(3 * fc.num_mortar, fc.num_mortar)) @ p["secondary_to_mortar_avg"]
                k.fr.append(SimpleNamespace(
                    m2p=csr(p["mortar_to_primary_int"]), p2m=csr(p["primary_to_mortar_avg"]),
                    m2s=csr(p["mortar_to_secondary_int"]), s2m=csr(p["secondary_to_mortar_avg"]),
                    m2p3=csr(sps.kron(p["mortar_to_primary_avg"], i3).tocsr()),
                    p2m3=csr(sps.kron(p["primary_to_mortar_int"], i3).tocsr()),
                    jump=csr(jump), traction=csr(trac), pressure_load=csr(pressure_load),
                    sel_n=csr(sel_n), sel_t=csr(sel_t), s2t=csr(s2t), coef=dev(fc.volumes * fc.kappa * 2.0),
                    div=csr(sps.csr_matrix(fc.sd.cell_faces.T)), vol=dev(np.asarray(fc.sd.cell_volumes, float)),
                    bc=None if fc.bc is None else {key: dev(v) for key, v in fc.bc.items() if not key.endswith("_type")}))
            self._const = k
        return self._const

    def _density(self, p):
        return ((p - self.fl.reference_pressure) * self.fl.compressibility).exp() * self.fl.density

    def _porosity(self, p, u, uj, k):
        dp = p - self.fl.reference_pressure
        b = k.ubc
        for j in range(len(self.fractures)):
            b = (k.fr[j].m2p3 @ uj[j]) + b
        return ((k.div_u @ u) + (k.div_u_b @ b) + (k.cons @ dp)) * k.inv_vol + dp * self.so.n_inv + self.so.reference_porosity

    def _fracture_flux(self, fc, q, p):
        """Darcy flux of a fracture: flux p (+ bound_flux p_b when the fracture carries boundary data)."""
        F = fc.data[DISCRETIZATION_MATRICES][self.fk]
        flux = ad.as_device_csr(F["flux"]) @ p
        if q.bc is not None:
            flux = flux + (ad.as_device_csr(F["bound_flux"]) @ q.bc["flow"])
        return flux

    def _advective(self, T, flux, weight, q, key):
        """Upwinded advective flux of a fracture (constitutive_laws.py:2555-2560) with its own boundary data, if any."""
        csr = ad.as_device_csr
        out = flux * (csr(T["transport"]) @ weight)
        if q.bc is not None:
            out = out + (csr(T["rhs_dir"]) @ (flux * q.bc[key])) + (csr(T["rhs_neu"]) @ q.bc[key])
        return out

    def _aperture(self, uj_j, q):
        return fn.maximum((q.sel_n @ (q.jump @ uj_j)) + self.so.residual_aperture, self.so.residual_aperture)

    def _group(self, parts):
        n = len(self.fractures)
        return parts[0], parts[1:1 + n], parts[1 + n], parts[2 + n:2 + 2 * n], parts[2 + 2 * n:2 + 3 * n], parts[2 + 3 * n:]

    def _parts(self, x):
        return self._group([x[self.offsets[q]:self.offsets[q + 1]] for q in range(len(self.sizes))])

    def update_discretizations(self, x) -> None:
        """What follows the iterate: the fracture flux discretization (aperture) and every upwind direction."""
        x = ad.device_vector(x)
        k = self._operands()
        p3, pf, _, _, lam, uj = self._parts(x)
        for j, fc in enumerate(self.fractures):
            self._discretize_fracture(fc, self._aperture(uj[j], k.fr[j]).cpu().numpy())
        mk = self.mobility_keyword
        b = k.bcq
        for j in range(len(self.fractures)):
            b = (k.fr[j].m2p @ lam[j]) + b
        q3 = ((k.F["flux"] @ p3) + (k.F["bound_flux"] @ b)).cpu().numpy()
        prm = self.data.setdefault(PARAMETERS, {}).setdefault(mk, {})
        prm["darcy_flux"], prm["bc"] = q3, self.bc["fluid_flux_type"]
        Upwind(mk).discretize(self.sd, self.data)
        for j, fc in enumerate(self.fractures):
            prm = fc.data.setdefault(PARAMETERS, {}).setdefault(mk, {})
            prm["darcy_flux"] = self._fracture_flux(fc, k.fr[j], pf[j]).cpu().numpy()
            prm["bc"] = fc.data[PARAMETERS][self.fk]["bc"] if fc.bc is None else fc.bc["fluid_flux_type"]
            Upwind(mk).discretize(fc.sd, fc.data)
            d = self._intf_data[j]
            d.setdefault(PARAMETERS, {}).setdefault(mk, {})["darcy_flux"] = lam[j].cpu().numpy()
            UpwindCoupling(mk).discretize(self.sd, fc.sd, SimpleNamespace(num_cells=fc.num_mortar), self.data, fc.data, d)

    def equations(self, x, x_prev, dt: float) -> list:
        k, ct, fl = self._operands(), self.ct, self.fl
        csr = ad.as_device_csr
        nfr = len(self.fractures)
        mk = self.mobility_keyword
        x, x_prev = ad.device_vector(x), ad.device_vector(x_prev)
        var = ad.variables([x[self.offsets[q]:self.offsets[q + 1]] for q in range(len(self.sizes))])
        p3, pf, u, t, lam, uj = self._group(var)
        p3n, pfn, un, _, _, ujn = self._parts(x_prev)
        w3 = self._density(p3) * (1.0 / fl.viscosity)
        wf = [self._density(pf[j]) * (1.0 / fl.viscosity) for j in range(nfr)]
        # interface mass fluxes, boundary operators of the matrix
        ifl, b_flow, b_mech = [], k.bcq, k.ubc
        for j in range(nfr):
            q = k.fr[j]
            U = self._intf_data[j][DISCRETIZATION_MATRICES][mk]
            ifl.append(lam[j] * ((csr(U["upwind_primary"]) @ (q.p2m @ (k.trace @ w3)))
                                 + (csr(U["upwind_secondary"]) @ (q.s2m @ wf[j]))))
            b_flow = (q.m2p @ lam[j]) + b_flow
            b_mech = (q.m2p3 @ uj[j]) + b_mech
        # ---- matrix: mass and momentum balance
        Tm = self.data[DISCRETIZATION_MATRICES][mk]
        q3 = (k.F["flux"] @ p3) + (k.F["bound_flux"] @ b_flow)
        neu = k.bcw
        for j in range(nfr):
            neu = (k.fr[j].m2p @ ifl[j]) + neu
        ff3 = q3 * (csr(Tm["transport"]) @ w3) + (csr(Tm["rhs_dir"]) @ (q3 * k.bcw)) + (csr(Tm["rhs_neu"]) @ neu)
        mass3 = (self._density(p3) * self._porosity(p3, u, uj, k) - self._density(p3n) * self._porosity(p3n, un, ujn, k)) \
            * (k.vol * (1.0 / dt)) + (k.div @ ff3)
        stress = (k.stress @ u) + (k.bound @ b_mech) + (k.grad_p @ (p3 - fl.reference_pressure))
        momentum = -(k.div3 @ stress)
        trace_p = (k.F["bound_pressure_cell"] @ p3) + (k.F["bound_pressure_face"] @ b_flow)
        mass_f, darcy, force, normal, tangential = [], [], [], [], []
        for j, fc in enumerate(self.fractures):
            q = k.fr[j]
            a, a_n = self._aperture(uj[j], q), self._aperture(ujn[j], q)
            # ---- fracture: mass balance
            Tf = fc.data[DISCRETIZATION_MATRICES][mk]
            qf = self._fracture_flux(fc, q, pf[j])
            mass_f.append((a * self._density(pf[j]) - a_n * self._density(pfn[j])) * (q.vol * (1.0 / dt))
                          + (q.div @ self._advective(Tf, qf, wf[j], q, "fluid_flux")) - (q.m2s @ ifl[j]))
            # ---- interface: Darcy law with the current aperture; force balance with the fluid pressure on the walls
            darcy.append(lam[j] - ((q.p2m @ trace_p) - (q.s2m @ pf[j])) * (q.s2m @ a.reciprocal()) * q.coef)
            force.append((q.p2m3 @ (stress * k.outward)) + (q.traction @ t[j]) + (q.pressure_load @ pf[j]))
            # ---- contact laws (porepy_b200.contact)
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
        return [mass3] + mass_f + [momentum] + darcy + force + normal + tangential

    def linearize(self, x, x_prev, dt: float):
        self.update_discretizations(x)
        return ad.assemble(self.equations(x, x_prev, dt))

    def time_step(self, x_prev, dt: float, linear_solver, tol: float = 1e-10, max_iterations: int = 30, verbose: bool = False):
        """Semismooth Newton; ``linear_solver(J, rhs) -> dx`` (e.g. ``contact.device_linear_solver(self)``).  Returns
        (x, history)."""
        import torch
        x_prev = ad.device_vector(x_prev)
        x = x_prev.clone()
        hist, r0 = [], None
        for it in range(max_iterations + 1):
            J, rhs = self.linearize(x, x_prev, dt)
            rn = float(torch.linalg.vector_norm(rhs))
            r0 = rn if r0 is None else r0
            hist.append({"iteration": it, "residual": rn})
            if verbose:
                print(hist[-1], flush=True)
            if rn <= tol * max(r0, 1e-300) or it == max_iterations:
                break
            x = x + linear_solver(J, rhs)
        return x, hist
