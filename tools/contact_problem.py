"""Generated frictional-contact problems of any size: ``FracturedMomentumBalance`` on a unit cube of hexahedra or
structured tetrahedra cut by planar fractures (``mdgrid.split_fractures`` + ``mdgrid.fracture_contacts``), with the
load cases and constants of tests/golden/contact_*.npz (west face fixed, east face displaced; stiffness with seeded
log-normal Lame parameters).  Used by the device-solve tests and tools/contact_solve_bench.py."""
from __future__ import annotations

import numpy as np

import porepy_b200 as pb
from porepy_b200 import mdgrid
from porepy_b200.contact import FracturedMomentumBalance

# the constants of tests/golden/contact_model.npz (the reference's defaults for that model)
SLIDING_CONSTANTS = dict(numerical_constant=1.0, characteristic_traction=27.0 / 7.0, friction_coefficient=0.4,
                         dilation_angle=0.1, reference_gap=1e-4, open_state_tolerance=1e-10)


def fracture_planes(g, planes: int):
    """``planes`` fractures x = const (evenly spaced grid planes), each covering the middle half in y and z."""
    n = int(round(1.0 / float(np.min(np.diff(np.unique(np.round(g.nodes[0], 12)))))))
    xs = sorted({int(round(n * (i + 1) / (planes + 1))) for i in range(planes)})
    if len(xs) != planes or xs[0] < 1 or xs[-1] > n - 1:
        raise ValueError(f"{planes} fracture planes do not fit a grid of {n} cells per side")
    lo, hi = np.floor(0.25 * n) / n, np.ceil(0.75 * n) / n
    return [mdgrid.faces_on_rectangle(g, 0, x / n, (lo, lo), (hi, hi)) for x in xs]


def generated_contact_problem(n: int, kind: str = "hex", planes: int = 1, seed: int = 0):
    """(problem, network): the sliding load case on n^3 hexahedra (``kind="hex"``) or the structured tetrahedra of n^3
    cubes (``kind="tet"``) with ``planes`` fractures."""
    g = pb.cart_grid_3d([n, n, n]) if kind == "hex" else pb.structured_tet_grid([n, n, n])
    net = mdgrid.split_fractures(g, fracture_planes(g, planes))
    m = net.matrix
    rng = np.random.default_rng(seed)
    C = pb.FourthOrderTensor(1.5 * np.exp(0.2 * rng.standard_normal(m.num_cells)),
                             2.0 * np.exp(0.2 * rng.standard_normal(m.num_cells)))
    bnd = np.asarray(m.tags["domain_boundary_faces"], bool)
    fc = m.face_centers
    west, east = bnd & (fc[0] < 1e-10), bnd & (fc[0] > 1 - 1e-10)
    bc = pb.BoundaryConditionVectorial(m, west | east, "dir")
    bc.internal_to_dirichlet(m)
    data = pb.initialize_data({}, "mechanics", {"fourth_order_tensor": C, "bc": bc})
    v = np.zeros((3, m.num_faces))
    v[0, east] = -0.01 * (1 + 0.3 * fc[2, east])           # compress across the fractures, unevenly
    v[1, east] = 0.02                                      # and shear them
    v[2, east] = 0.005 * fc[1, east]
    prob = FracturedMomentumBalance(m, data, v.ravel("F"), mdgrid.fracture_contacts(net), SLIDING_CONSTANTS)
    return prob, net
