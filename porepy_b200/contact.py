"""Frictional contact on fractures, the reference's ``pp.MomentumBalance`` on the device AD chain -- the contact part of
BASELINE config[4]: MPSA elasticity in the 3-D matrix (``porepy_b200.Mpsa``; the two sides of every fracture are internal
Dirichlet boundaries carrying the interface displacement), force balance on the matrix-fracture interfaces and the
semismooth complementarity laws of the contact traction.

Unknowns: [u (3 per matrix cell) | t (contact traction, 3 per fracture cell, in the fracture's local frame: two tangential
components, then the normal one; scaled by the characteristic traction) | u_j (3 per mortar cell)];
equations, in the reference's order:

* ``momentum_balance_equation``        -div_nd (stress u + bound_stress (u_b + Pi^avg u_j)) - f          models/momentum_balance.py
* ``interface_force_balance_equation`` Pi^int (n_out . sigma) + vol S Pi^int R^T t T_c                    momentum_balance.py:127-183,
                                                                                               constitutive_laws.py:2956-3001
* ``normal_fracture_deformation_equation``      t_n + max(-t_n - c ([u]_n - g), 0),   g = g0 + tan(psi) ||[u]_t||
                                                                                               contact_mechanics.py:80-129
* ``tangential_fracture_deformation_equation``  (1 - chi) (b_p s - max(b_p, ||s||) t_t) + chi t_t,
                                       s = t_t + c ([u]_t - [u]_t^n),  b_p = max(-mu_f t_n, 0),  chi = 1 where b_p <= tol
                                                                                               contact_mechanics.py:131-245

with the displacement jump ``[u] = R Pi^avg_{mortar -> fracture} S u_j`` (``S``: side signs, ``R``: global -> local
coordinates; constitutive_laws.py ``displacement_jump``).  ``maximum`` / ``l2_norm`` / ``characteristic_function`` are those of
``porepy_b200.ad_functions`` with the reference's tie rules, so the Jacobian of the semismooth laws is the reference's.  The
elastic fracture-deformation laws (Barton-Bandis closure, tangential stiffness) are off in the reference's defaults and not
stated here.  The Jacobian has zeros on the diagonal of the complementarity rows, so point and 3 x 3 Jacobi are undefined:
``device_linear_solver`` solves the Newton steps on the device with restarted GMRES preconditioned by the inverses of the
local blocks of ``block_layout`` (one per matrix cell, one per fracture cell with its two mortar cells); ``time_step``
takes any ``linear_solver(J, rhs) -> dx``.
``tests/golden/contact_model.npz`` pins Jacobian, residual, residual history and the converged sliding state.
"""
from __future__ import annotations

from types import SimpleNamespace

import numpy as np
import scipy.sparse as sps

from . import ad, ad_functions as fn
from .fv import Mpsa
from .params import DISCRETIZATION_MATRICES


class FractureContact:
    """One fracture and its two-sided interface: ``mortar_to_primary_avg``, ``primary_to_mortar_int`` (faces of the matrix
    grid), ``mortar_to_secondary_avg``, ``secondary_to_mortar_int`` (cells of the fracture): the SCALAR projections of the
    reference's ``MortarGrid``; ``mortar_sign`` (+-1 per mortar cell: ``sign_of_mortar_sides``), ``mortar_volumes``,
    ``local_coordinates`` (3 nfc x 3 nfc, rows per cell: tangent, tangent, normal)."""

    def __init__(self, mortar_to_primary_avg, primary_to_mortar_int, mortar_to_secondary_avg, secondary_to_mortar_int,
                 mortar_sign, mortar_volumes, local_coordinates):
        i3 = sps.identity(3, format="csr")
        self.m2p = sps.kron(sps.csr_matrix(mortar_to_primary_avg), i3).tocsr()
        self.p2m = sps.kron(sps.csr_matrix(primary_to_mortar_int), i3).tocsr()
        self.m2s = sps.kron(sps.csr_matrix(mortar_to_secondary_avg), i3).tocsr()
        self.s2m = sps.kron(sps.csr_matrix(secondary_to_mortar_int), i3).tocsr()
        self.sign = sps.diags(np.repeat(np.asarray(mortar_sign, float), 3)).tocsr()
        self.volumes = np.repeat(np.asarray(mortar_volumes, float), 3)
        self.rotation = sps.csr_matrix(local_coordinates)
        self.num_mortar = int(np.asarray(mortar_sign).size)
        self.num_cells = int(self.rotation.shape[0] // 3)
        self.mortar_to_secondary = sps.csr_matrix(mortar_to_secondary_avg)


def mortar_pairs(mortar_to_secondary) -> np.ndarray:
    """(num fracture cells, 2): the two mortar cells of every fracture cell, from the scalar mortar -> fracture
    projection.  A fracture cell without exactly two mortar cells (an intersection, a one-sided interface) has no
    local block of the kind ``local_block_layout`` builds."""
    m2s = sps.csr_matrix(mortar_to_secondary, copy=True)
    m2s.eliminate_zeros()
    m2s.sort_indices()
    if np.any(np.diff(m2s.indptr) != 2):
        raise NotImplementedError("local blocks need exactly two mortar cells per fracture cell")
    return m2s.indices.reshape(-1, 2).astype(np.int64)


def local_block_layout(num_cells: int, pairs, cell_unknowns, cell_equations, fracture_unknowns, fracture_equations):
    """The local blocks of a contact model's Jacobian, from the model's own offsets: one block per matrix cell (its
    ``cell_unknowns`` / ``cell_equations``: lists of (offset, width): entries offset + width * cell + 0..width-1) and one
    per fracture cell (``fracture_unknowns[j]`` / ``fracture_equations[j]`` of fracture j: lists of (offset, width, on),
    ``on`` = "fracture" for a field per fracture cell, "mortar" for a field per mortar cell: both mortar cells of the
    fracture cell, ``pairs[j]``, go into its block).  Returns ``SimpleNamespace(ptr, rows, cols)``: every row and every
    column of the Jacobian belongs to exactly one block (asserted)."""
    def take(fields, ids_of):
        return np.hstack([(off + ids_of[on][:, :, None] * w + np.arange(w)).reshape(ids_of[on].shape[0], -1)
                          for off, w, on in fields])
    cells = {"cell": np.arange(num_cells, dtype=np.int64)[:, None]}
    rows = [take([(o, w, "cell") for o, w in cell_equations], cells)]
    cols = [take([(o, w, "cell") for o, w in cell_unknowns], cells)]
    for pr, fu, fe in zip(pairs, fracture_unknowns, fracture_equations):
        pr = np.asarray(pr, np.int64)
        ids = {"fracture": np.arange(pr.shape[0], dtype=np.int64)[:, None], "mortar": pr}
        rows.append(take(fe, ids))
        cols.append(take(fu, ids))
    for r, c in zip(rows, cols):
        assert r.shape == c.shape, "a block needs as many equations as unknowns"
    sizes = np.concatenate([np.full(r.shape[0], r.shape[1], np.int64) for r in rows])
    layout = SimpleNamespace(ptr=np.concatenate(([0], np.cumsum(sizes))).astype(np.int64),
                             rows=np.concatenate([r.ravel() for r in rows]), cols=np.concatenate([c.ravel() for c in cols]))
    n = layout.rows.size
    assert np.array_equal(np.bincount(layout.rows, minlength=n), np.ones(n, np.int64)), "rows: not a bijection"
    assert np.array_equal(np.bincount(layout.cols, minlength=n), np.ones(n, np.int64)), "columns: not a bijection"
    return layout


def offsets_of(sizes) -> np.ndarray:
    return np.concatenate(([0], np.cumsum(sizes))).astype(np.int64)


class DeviceLinearSolver:
    """``linear_solver(J, rhs) -> dx`` of the models' ``time_step`` on the device: the local blocks of ``J``
    (``problem.block_layout()``, uploaded on the first call) are inverted at every call and GMRES
    (``krylov.gmres``) runs with them as right preconditioner; its info goes to ``history``.  Raises ``RuntimeError``
    when GMRES does not reach ``tol``."""

    def __init__(self, problem, tol: float = 1e-12, restart: int = 100, maxiter: int = 2000):
        self.layout = problem.block_layout()
        self.tol, self.restart, self.maxiter = float(tol), int(restart), int(maxiter)
        self.blocks = None
        self.history = []

    def __call__(self, J, rhs):
        from . import krylov
        if self.blocks is None:
            self.blocks = krylov.LocalBlocks(self.layout)
        self.blocks.factor(J)
        dx, info = krylov.gmres(J, rhs, precond=self.blocks, tol=self.tol, restart=self.restart, maxiter=self.maxiter)
        self.history.append(info)
        if not info["converged"]:
            raise RuntimeError(f"GMRES did not converge: {info['iterations']} iterations, relative residual "
                               f"{info['relres']:.3e} (tol {self.tol:.1e})")
        return dx


def device_linear_solver(problem, tol: float = 1e-12, restart: int = 100, maxiter: int = 2000) -> DeviceLinearSolver:
    """The device solve of the Newton steps of ``problem`` (a contact model with ``block_layout()``), for its
    ``time_step(..., linear_solver=...)``."""
    return DeviceLinearSolver(problem, tol, restart, maxiter)


class FracturedMomentumBalance:
    """``sd``: the 3-D matrix grid (faces split along the fractures, ``fracture_faces`` tag), ``data``:
    ``parameters[keyword]`` with ``fourth_order_tensor`` and the vectorial ``bc`` (fracture faces Dirichlet,
    ``internal_to_dirichlet``); ``bc_values``: 3 nf face-major (displacement / traction); ``fractures``: list of
    ``FractureContact``; ``constants``: ``numerical_constant, characteristic_traction, friction_coefficient,
    dilation_angle, reference_gap, open_state_tolerance``."""

    def __init__(self, sd, data: dict, bc_values, fractures, constants: dict, body_force=None, keyword: str = "mechanics"):
        if int(sd.dim) != 3:
            raise NotImplementedError("a 3-D matrix grid is expected")
        self.sd, self.data, self.kw = sd, data, keyword
        self.bc_values = np.asarray(bc_values, float)
        self.fractures = list(fractures)
        self.k = SimpleNamespace(**{k: float(v) for k, v in constants.items()})
        self.nc, self.nf = int(sd.num_cells), int(sd.num_faces)
        self.body_force = np.zeros(3 * self.nc) if body_force is None else np.asarray(body_force, float)
        nt = [3 * f.num_cells for f in self.fractures]
        nj = [3 * f.num_mortar for f in self.fractures]
        self.sizes = [3 * self.nc] + nt + nj
        self.offsets = np.concatenate(([0], np.cumsum(self.sizes))).astype(np.int64)
        self._const = None

    @property
    def num_dofs(self) -> int:
        return int(self.offsets[-1])

    def discretize(self) -> None:
        Mpsa(self.kw).discretize(self.sd, self.data)
        self._const = None

    def block_layout(self):
        """Local blocks of the Jacobian: u of every matrix cell (3), and per fracture cell its traction with the u_j of
        its two mortar cells (9), paired with the momentum balance, resp. the normal and tangential laws and the two
        force balances."""
        nfr = len(self.fractures)
        o = self.offsets
        e = offsets_of([3 * self.nc] + [3 * f.num_mortar for f in self.fractures] + [f.num_cells for f in self.fractures]
                       + [2 * f.num_cells for f in self.fractures])
        return local_block_layout(
            self.nc, [mortar_pairs(f.mortar_to_secondary) for f in self.fractures], [(o[0], 3)], [(e[0], 3)],
            [[(o[1 + j], 3, "fracture"), (o[1 + nfr + j], 3, "mortar")] for j in range(nfr)],
            [[(e[1 + nfr + j], 1, "fracture"), (e[1 + 2 * nfr + j], 2, "fracture"), (e[1 + j], 3, "mortar")]
             for j in range(nfr)])

    def _operands(self):
        if self._const is None:
            csr, dev = ad.as_device_csr, ad.device_vector
            M = self.data[DISCRETIZATION_MATRICES][self.kw]
            cf = sps.csr_matrix(self.sd.cell_faces)
            frac = np.asarray(self.sd.tags["fracture_faces"], bool)
            out = np.where(frac, np.asarray(cf.sum(axis=1)).ravel(), 0.0)      # +-1 on fracture faces: outward normal
            k = SimpleNamespace(
                div3=csr(sps.kron(sps.csr_matrix(self.sd.cell_faces.T), sps.identity(3)).tocsr()),
                stress=csr(M["stress"]), bound=csr(M["bound_stress"]),
                outward=dev(np.repeat(out, 3)), f=dev(self.body_force), fr=[])
            k.stress_b = k.bound @ dev(self.bc_values)
            for fc in self.fractures:
                n = fc.num_cells
                sel_n = sps.csr_matrix((np.ones(n), (np.arange(n), 3 * np.arange(n) + 2)), shape=(n, 3 * n))
                sel_t = sps.csr_matrix((np.ones(2 * n), (np.arange(2 * n), 3 * np.repeat(np.arange(n), 2)
                                                         + np.tile([0, 1], n))), shape=(2 * n, 3 * n))
                s2t = sps.csr_matrix((np.ones(2 * n), (np.arange(2 * n), np.repeat(np.arange(n), 2))), shape=(2 * n, n))
                jump = fc.rotation @ fc.m2s @ fc.sign                            # u_j -> local displacement jump
                trac = sps.diags(fc.volumes * self.k.characteristic_traction) @ fc.sign @ fc.s2m @ fc.rotation.T
                k.fr.append(SimpleNamespace(m2p=csr(fc.m2p), p2m=csr(fc.p2m), jump=csr(jump), traction=csr(trac),
                                            sel_n=csr(sel_n), sel_t=csr(sel_t), s2t=csr(s2t)))
            self._const = k
        return self._const

    def equations(self, x, x_prev) -> list:
        k, c = self._operands(), self.k
        nfr = len(self.fractures)
        x, x_prev = ad.device_vector(x), ad.device_vector(x_prev)
        var = ad.variables([x[self.offsets[q]:self.offsets[q + 1]] for q in range(len(self.sizes))])
        u, t, uj = var[0], var[1:1 + nfr], var[1 + nfr:]
        ujn = [x_prev[self.offsets[1 + nfr + j]:self.offsets[2 + nfr + j]] for j in range(nfr)]
        boundary = None
        for j in range(nfr):
            term = k.fr[j].m2p @ uj[j]
            boundary = term if boundary is None else boundary + term
        stress = (k.stress @ u) + k.stress_b
        if boundary is not None:
            stress = stress + (k.bound @ boundary)
        momentum = -(k.div3 @ stress) - k.f
        force, normal, tangential = [], [], []
        for j in range(nfr):
            q = k.fr[j]
            force.append((q.p2m @ (stress * k.outward)) + (q.traction @ t[j]))
            jump, jump_n = q.jump @ uj[j], q.jump @ ujn[j]
            t_n, u_n = q.sel_n @ t[j], q.sel_n @ jump
            t_t, u_t, u_t_prev = q.sel_t @ t[j], q.sel_t @ jump, q.sel_t @ jump_n
            gap = fn.l2_norm(2, u_t) * float(np.tan(c.dilation_angle)) + c.reference_gap
            normal.append(t_n + fn.maximum(-t_n - (u_n - gap) * c.numerical_constant, 0.0))
            s = t_t + (u_t - u_t_prev) * c.numerical_constant
            b_p = fn.maximum(t_n * (-c.friction_coefficient), 0.0)
            chi = q.s2t @ fn.characteristic_function(c.open_state_tolerance, b_p).val
            tangential.append(((q.s2t @ b_p) * s - (q.s2t @ fn.maximum(b_p, fn.l2_norm(2, s))) * t_t) * (1.0 - chi)
                              + t_t * chi)
        return [momentum] + force + normal + tangential

    def linearize(self, x, x_prev):
        """(J as ``DeviceCsr``, -R as a CUDA tensor) at the iterate ``x`` (previous time step ``x_prev``)."""
        return ad.assemble(self.equations(x, x_prev))

    def time_step(self, x_prev, linear_solver, x0=None, tol: float = 1e-10, max_iterations: int = 30, verbose: bool = False):
        """Semismooth Newton from ``x0`` (default: the previous state); ``linear_solver(J, rhs) -> dx``, e.g.
        ``device_linear_solver(self)``."""
        import torch
        x_prev = ad.device_vector(x_prev)
        x = x_prev.clone() if x0 is None else ad.device_vector(x0).clone()
        hist, r0 = [], None
        for it in range(max_iterations + 1):
            J, rhs = self.linearize(x, x_prev)
            rn = float(torch.linalg.vector_norm(rhs))
            r0 = rn if r0 is None else r0
            hist.append({"iteration": it, "residual": rn})
            if verbose:
                print(hist[-1], flush=True)
            if rn <= tol * max(r0, 1e-300) or it == max_iterations:
                break
            x = x + linear_solver(J, rhs)
        return x, hist
