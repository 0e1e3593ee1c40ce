"""Synthetic mixed-dimensional meshes: a 3-D grid cut by planar, mutually disjoint fractures.

The reference builds fracture networks with its meshing package (fracs/: ``split_grid``, ``meshing.cart_grid`` /
``create_mdg``), which -- like the reference itself -- is absent on the GPU box.  This module produces, from one of the
generators of ``porepy_b200.grid`` (hexahedra or structured tetrahedra) and sets of interior faces lying in a plane, what
the hot path consumes of such a network: the 3-D grid with faces and nodes duplicated along the fractures (``fracture_faces``
tag, one side per copy), one 2-D grid per fracture embedded in 3-D (cells = the fracture faces; boundary edges tagged as
tips) and, per fracture, the four mortar projections of a matching two-sided interface (``MortarGrid``:
grids/mortar_grid.py) in the form ``porepy_b200.mdflow.MdInterface`` takes.  Intersecting fractures (1-D / 0-D subdomains)
are covered by the reference-generated fixtures, not by this generator.  O(n) NumPy, run once per mesh; not the hot path.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import scipy.sparse as sps
from scipy.sparse.csgraph import connected_components

from .grid import Grid


def faces_on_rectangle(g: Grid, axis: int, at: float, lo, hi, tol: float = 1e-9) -> np.ndarray:
    """Interior faces of ``g`` lying in the plane ``x_axis = at`` whose centres fall inside [lo, hi] in the two other
    coordinates (each a pair)."""
    fc = g.face_centers
    others = [a for a in range(3) if a != axis]
    two_cells = np.asarray(abs(g.cell_faces).sum(axis=1)).ravel() == 2
    nrm = g.face_normals / np.maximum(g.face_areas, 1e-300)
    sel = (np.abs(fc[axis] - at) < tol) & (np.abs(np.abs(nrm[axis]) - 1.0) < 1e-6) & two_cells
    for a, l, h in zip(others, lo, hi):
        sel &= (fc[a] > l - tol) & (fc[a] < h + tol)
    return np.flatnonzero(sel)


@dataclass
class FractureNetwork:
    matrix: Grid                 # 3-D grid, split
    fractures: list              # 2-D grids
    interfaces: list             # per fracture: dict of the four projections + mortar cell volumes
    sides: list                  # per fracture: (faces of side 0, faces of side 1) in the split 3-D grid


def _loops(g: Grid, faces: np.ndarray):
    ip, ix = g.face_nodes.indptr, g.face_nodes.indices
    n = np.diff(ip)[faces]
    if n.size == 0 or np.any(n != n[0]):
        raise ValueError("the faces of one fracture must have the same number of nodes")
    L = int(n[0])
    return ix[(ip[faces][:, None] + np.arange(L)[None, :])], L


def split_fractures(g: Grid, fracture_faces) -> FractureNetwork:
    """Cut the 3-D grid ``g`` (with geometry) along the given face sets; see the module docstring."""
    if g.dim != 3:
        raise ValueError("a 3-D grid is expected")
    fracture_faces = [np.asarray(f, dtype=np.int64) for f in fracture_faces]
    nf, nc, nn = g.num_faces, g.num_cells, g.num_nodes
    all_ff = np.concatenate(fracture_faces) if fracture_faces else np.zeros(0, np.int64)
    if np.unique(all_ff).size != all_ff.size:
        raise ValueError("fractures must not share faces")
    cf = sps.coo_matrix(g.cell_faces)
    if np.any(np.bincount(cf.row, minlength=nf)[all_ff] != 2):
        raise ValueError("fracture faces must be interior faces")
    is_ff = np.zeros(nf, bool)
    is_ff[all_ff] = True
    # ---- 1. every fracture face f keeps its +1 cell; a copy f' (same nodes, same normal) takes the -1 cell
    copy_of = np.full(nf, -1, np.int64)
    copy_of[all_ff] = nf + np.arange(all_ff.size)
    rows = cf.row.astype(np.int64).copy()
    cols = cf.col.astype(np.int64)
    dat = cf.data.astype(np.float64)
    moved = is_ff[rows] & (dat < 0)
    rows[moved] = copy_of[rows[moved]]
    nf2 = nf + all_ff.size
    orig_face = np.concatenate((np.arange(nf), all_ff))
    # ---- 2. split the nodes: around a fracture node, cells connected through non-fracture faces share a copy
    fip, fix = g.face_nodes.indptr, g.face_nodes.indices
    fnode = np.zeros(nn, bool)
    if all_ff.size:
        cnt_f = np.diff(fip)[all_ff]
        pos = np.repeat(fip[all_ff], cnt_f) + (np.arange(cnt_f.sum()) - np.repeat(np.cumsum(cnt_f) - cnt_f, cnt_f))
        fnode[fix[pos]] = True
    # fractures that touch would need their intersection line as a 1-D subdomain: not generated here
    owner = np.full(nn, -1, np.int64)
    for k, F in enumerate(fracture_faces):
        cf_ = np.diff(fip)[F]
        pk = np.repeat(fip[F], cf_) + (np.arange(cf_.sum()) - np.repeat(np.cumsum(cf_) - cf_, cf_))
        nk = np.unique(fix[pk])
        if np.any((owner[nk] >= 0) & (owner[nk] != k)):
            raise ValueError("fractures must not share nodes (intersecting fractures are not supported by this generator)")
        owner[nk] = k
    # (new face row, cell, node) triples restricted to fracture nodes
    cnt = np.diff(fip)[orig_face[rows]]
    t_face = np.repeat(rows, cnt)
    t_cell = np.repeat(cols, cnt)
    start = np.repeat(fip[orig_face[rows]], cnt)
    within = np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    t_node = fix[start + within]
    keep = fnode[t_node]
    kf, kc, kn = t_face[keep], t_cell[keep], t_node[keep]
    pair_key = kc * nn + kn
    upair, pinv = np.unique(pair_key, return_inverse=True)
    # edges between the two (cell, node) pairs of every non-fracture interior face
    nonfrac = ~is_ff[orig_face[kf]]
    ek = kf[nonfrac] * nn + kn[nonfrac]
    o = np.argsort(ek, kind="stable")
    eks, ep = ek[o], pinv[nonfrac][o]
    same = eks[1:] == eks[:-1]
    a, b = ep[:-1][same], ep[1:][same]
    graph = sps.coo_matrix((np.ones(a.size), (a, b)), shape=(upair.size, upair.size))
    _, comp = connected_components(graph, directed=False)
    pnode = upair % nn
    # per node: the component holding the smallest pair keeps the node, every other component gets a copy
    order = np.lexsort((comp, pnode))
    pn, pc = pnode[order], comp[order]
    first_of_node = np.r_[True, pn[1:] != pn[:-1]]
    new_comp = np.r_[True, (pn[1:] != pn[:-1]) | (pc[1:] != pc[:-1])]
    extra = new_comp & ~first_of_node
    copy_id = np.cumsum(extra) - 1 + nn                 # id of the latest copy created so far
    # within one node the components come sorted: the first keeps pn, later ones take the running copy id
    grp = np.cumsum(new_comp) - 1
    grp_first = np.flatnonzero(new_comp)
    grp_node = np.where(first_of_node[grp_first], pn[grp_first], copy_id[grp_first])
    node_of_pair = np.empty(upair.size, np.int64)
    node_of_pair[order] = grp_node[grp]
    n_extra = int(extra.sum())
    orig_node = np.concatenate((np.arange(nn), pn[extra]))
    # ---- face -> nodes of the split grid (loop order kept): the nodes seen from the face's first cell
    new_node = t_node.copy()
    new_node[keep] = node_of_pair[pinv]
    o2 = np.argsort(t_face, kind="stable")
    tf, tc, tn = t_face[o2], t_cell[o2], new_node[o2]
    first_cell = np.full(nf2, -1, np.int64)
    firsts = np.r_[True, tf[1:] != tf[:-1]]
    first_cell[tf[firsts]] = tc[firsts]
    sel = tc == first_cell[tf]
    tf, tn = tf[sel], tn[sel]
    cnt2 = np.bincount(tf, minlength=nf2)
    fn2 = sps.csc_matrix((np.ones(tn.size, bool), tn, np.concatenate(([0], np.cumsum(cnt2)))),
                         shape=(nn + n_extra, nf2))
    cf2 = sps.csc_matrix(sps.coo_matrix((dat, (rows, cols)), shape=(nf2, nc)))
    cf2.sort_indices()
    m = Grid(3, g.nodes[:, orig_node], fn2, cf2, name=g.name)
    m.set_geometry(g.face_normals[:, orig_face], g.face_centers[:, orig_face], g.face_areas[orig_face],
                   g.cell_centers, g.cell_volumes)
    m.tags["domain_boundary_faces"] = np.concatenate((g.tags["domain_boundary_faces"], np.zeros(all_ff.size, bool)))
    m.tags["fracture_faces"] = np.concatenate((is_ff, np.ones(all_ff.size, bool)))
    m.tags["tip_faces"] = np.zeros(nf2, bool)
    if hasattr(g, "cart_dims"):
        m.cart_dims = g.cart_dims
    # ---- 3. the fracture planes as 2-D grids and their interfaces
    lo, hi = g.nodes.min(axis=1), g.nodes.max(axis=1)
    fractures, interfaces, sides = [], [], []
    for F in fracture_faces:
        loops, L = _loops(g, F)
        un, linv = np.unique(loops.ravel(), return_inverse=True)
        loc = linv.reshape(-1, L)
        ea, eb = loc.ravel(), np.roll(loc, -1, axis=1).ravel()
        ekey = np.minimum(ea, eb) * un.size + np.maximum(ea, eb)
        ue, first, einv = np.unique(ekey, return_index=True, return_inverse=True)
        en = np.stack((ue // un.size, ue % un.size), axis=1)
        ne, mcells = ue.size, F.size
        nodes2 = g.nodes[:, un]
        pa, pb_ = nodes2[:, en[:, 0]], nodes2[:, en[:, 1]]
        nu = g.face_normals[:, F[0]] / g.face_areas[F[0]]
        enrm = np.cross((pb_ - pa).T, nu).T
        ec = 0.5 * (pa + pb_)
        cc = g.face_centers[:, F]
        cell_of = np.repeat(np.arange(mcells), L)
        sgn = np.sign(np.einsum("ij,ij->j", enrm[:, einv], ec[:, einv] - cc[:, cell_of]))
        cfk = sps.csc_matrix(sps.coo_matrix((sgn, (einv, cell_of)), shape=(ne, mcells)))
        cfk.sort_indices()
        fnk = sps.csc_matrix((np.ones(2 * ne, bool), en.ravel(), np.arange(0, 2 * ne + 1, 2)), shape=(un.size, ne))
        fg = Grid(2, nodes2, fnk, cfk, name="Fracture")
        # a boundary edge's stored normal must point out of its only cell when that entry is +1: already so by the sign
        fg.set_geometry(enrm, ec, np.linalg.norm(pb_ - pa, axis=0), cc, g.face_areas[F])
        one_cell = np.asarray(abs(cfk).sum(axis=1)).ravel() == 1
        on_bbox = np.any((np.abs(ec - lo[:, None]) < 1e-12) | (np.abs(ec - hi[:, None]) < 1e-12), axis=0)
        fg.tags["domain_boundary_faces"] = one_cell & on_bbox
        fg.tags["tip_faces"] = one_cell & ~on_bbox
        fg.tags["fracture_faces"] = np.zeros(ne, bool)
        fractures.append(fg)
        s0, s1 = F, copy_of[F]
        sides.append((s0, s1))
        idx = np.arange(mcells)
        m2p = sps.csr_matrix((np.ones(2 * mcells), (np.concatenate((s0, s1)), np.arange(2 * mcells))),
                             shape=(nf2, 2 * mcells))
        m2s = sps.csr_matrix((np.ones(2 * mcells), (np.concatenate((idx, idx)), np.arange(2 * mcells))),
                             shape=(mcells, 2 * mcells))
        interfaces.append(dict(mortar_to_primary_int=m2p, primary_to_mortar_avg=m2p.T.tocsr(),
                               mortar_to_secondary_int=m2s, secondary_to_mortar_avg=m2s.T.tocsr(),
                               cell_volumes=np.concatenate((g.face_areas[F], g.face_areas[F]))))
    return FractureNetwork(m, fractures, interfaces, sides)


def mortar_signs(g: Grid, mortar_to_primary) -> np.ndarray:
    """+-1 per mortar cell: the orientation of its primary face seen from the matrix cell on that side (the face
    normal points out of that cell: +1), as the reference's ``sign_of_mortar_sides``.  ``mortar_to_primary``: faces x
    mortar cells, one face per mortar cell."""
    m2p = sps.csc_matrix(mortar_to_primary)
    m2p.eliminate_zeros()
    if np.any(np.diff(m2p.indptr) != 1):
        raise ValueError("every mortar cell needs exactly one primary face")
    faces = m2p.indices
    return np.asarray(sps.csr_matrix(g.cell_faces)[faces].sum(axis=1)).ravel().astype(float)


def tangent_normal_basis(normal) -> np.ndarray:
    """Rows: tangent, tangent, normal of the unit ``normal`` (3,): the first tangent is n rotated by 90 degrees in the two
    coordinates other than n's largest one (ascending), or the unit vector of the first of them when n is aligned with an
    axis; the second is n x t1.  The reference's ``TangentialNormalProjection`` convention."""
    n = np.asarray(normal, float) / np.linalg.norm(normal)
    i = int(np.argmax(np.abs(n)))
    a, b = [q for q in range(3) if q != i]
    t1 = np.zeros(3)
    if np.hypot(n[a], n[b]) < 1e-8:
        t1[a] = 1.0
    else:
        t1[a], t1[b] = -n[b], n[a]
    t1 /= np.linalg.norm(t1)
    t2 = np.cross(n, t1)
    t2 /= np.linalg.norm(t2)
    return np.linalg.inv(np.column_stack((t1, t2, n)))


def fracture_local_coordinates(g: Grid, mortar_to_primary, mortar_sign, num_cells: int) -> sps.csr_matrix:
    """3 nfc x 3 nfc rotation to the local frame of a planar fracture, the same frame in every fracture cell.  The normal
    is the outward unit normal of the matrix cell on the mortar side of sign -1: it points from that side across the
    fracture, so that the normal component of the jump ``sum(sign * u_j)`` (the +1 side minus the -1 side) is positive
    when the fracture opens.  (The reference takes the side of its first mortar cell, which has sign -1 in its split
    grids, where the original face keeps the cell it points into.)"""
    m2p = sps.csc_matrix(mortar_to_primary)
    m2p.eliminate_zeros()
    sign = np.asarray(mortar_sign, float)
    neg = np.flatnonzero(sign < 0)
    if neg.size == 0:
        raise ValueError("a two-sided interface needs mortar cells of sign -1")
    f0 = int(m2p.indices[m2p.indptr[neg[0]]])
    n = -np.asarray(g.face_normals)[:, f0] / float(np.asarray(g.face_areas)[f0])
    return sps.kron(sps.identity(int(num_cells)), sps.csr_matrix(tangent_normal_basis(n))).tocsr()


def fracture_contacts(net: FractureNetwork) -> list:
    """``contact.FractureContact`` of every (planar) fracture of a network from ``split_fractures``: the projections of
    the matching two-sided interface (one mortar cell per fracture face and side: the ``*_avg`` and ``*_int`` forms
    coincide), the mortar signs and the local frame by the reference's conventions."""
    from .contact import FractureContact
    out = []
    for fg, intf in zip(net.fractures, net.interfaces):
        m2p = intf["mortar_to_primary_int"]
        sign = mortar_signs(net.matrix, m2p)
        out.append(FractureContact(m2p, m2p.T.tocsr(), intf["mortar_to_secondary_int"],
                                   intf["secondary_to_mortar_avg"], sign, intf["cell_volumes"],
                                   fracture_local_coordinates(net.matrix, m2p, sign, fg.num_cells)))
    return out
