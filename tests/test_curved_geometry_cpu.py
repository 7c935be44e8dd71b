"""CPU: second-order (27-node) geometry -- the reference's convergence orders, the 27-node ghost-layer builder
(pmgx_ghostmesh_create_q2) and its input checks.

Order thresholds, calibrated with tests/curved_reference.py on the annular sector (P4, exact volume 3 pi / 4):
  volume error   Q1 geometry 2.35e-1, 6.01e-2, 1.51e-2 at n = 2, 4, 8 (order 1.97, 1.99)
                 Q2 geometry 1.83e-3, 1.16e-4, 7.29e-6                 (order 3.98, 3.99)
  nodal error    Q1 geometry 3.25e-1, 1.11e-1, 2.97e-2 at n = 2, 4, 8 (order 1.55, 1.91)
                 Q2 geometry 4.29e-3, 2.81e-4, 1.78e-5                 (order 3.93, 3.98)
The tests ask for a Q2 order above 3.5 and at least 1.5 above the Q1 order: about halfway between the two."""
import ctypes
import itertools

import numpy as np
import pytest
from scipy.spatial import cKDTree

from oracle import mesh as om
import curved_reference as cr

Q2_MIN_ORDER, MIN_GAIN = 3.5, 1.5


def orders(f, meshes):
    e = [f(m) for m in meshes]
    return np.log2(e[0] / e[1])


def test_volume_order_exceeds_trilinear():
    exact = 0.75 * np.pi
    q2 = [cr.q2_box(n, n, n, cr.sector) for n in (4, 8)]
    o2 = orders(lambda m: abs(cr.volume(m) - exact), q2)
    o1 = orders(lambda m: abs(cr.volume(m.corners()) - exact), q2)
    assert o2 > Q2_MIN_ORDER and o2 > o1 + MIN_GAIN, (o1, o2)


def test_nodal_error_order_exceeds_trilinear():
    q2 = [cr.q2_box(n, n, n, cr.sector) for n in (2, 4)]
    o2 = orders(cr.nodal_error, q2)
    o1 = orders(lambda m: cr.nodal_error(m.corners()), q2)
    assert o2 > Q2_MIN_ORDER and o2 > o1 + MIN_GAIN, (o1, o2)


def test_trilinear_nodes_reproduce_q1_geometry():
    m = om.create_box(3, 2, 4, perturb=0.2)
    q = cr.q2_from_q1(m)
    from oracle import operator as oo
    for P in (1, 4):
        G1, _ = oo.geometry_factors(m.verts, m.geom_dofmap, P)
        G2, _ = cr.geometry_factors(q.verts, q.geom_dofmap, P)
        assert np.abs(G2 - G1).max() <= 1e-13 * np.abs(G1).max()
        assert np.abs(cr.dof_coords(q, P) - om.dof_coords(m, P)).max() < 1e-14


def _rotations():
    out = []
    for perm in itertools.permutations(range(3)):
        for flips in itertools.product((0, 1), repeat=3):
            M = np.zeros((3, 3))
            for d in range(3):
                M[d, perm[d]] = -1.0 if flips[d] else 1.0
            if np.linalg.det(M) > 0:
                out.append((perm, flips))
    return out


def scrambled_q2(q, seed, nranks):
    """q with its nodes renumbered, its cells shuffled and every cell's frame rotated (all 27 nodes), and a skew
    partition into nranks parts."""
    rng = np.random.default_rng(seed)
    nn, nc = len(q.verts), q.ncells
    vnew = rng.permutation(nn)
    coords = np.empty_like(q.verts)
    coords[vnew] = q.verts
    rots = _rotations()
    cells = np.empty((nc, 27), dtype=np.int64)
    for c in range(nc):
        perm, flips = rots[rng.integers(24)]
        for new in itertools.product(range(3), repeat=3):
            old = [2 - new[perm[d]] if flips[d] else new[perm[d]] for d in range(3)]
            cells[c, 9 * new[0] + 3 * new[1] + new[2]] = vnew[q.geom_dofmap[c, 9 * old[0] + 3 * old[1] + old[2]]]
    cells = cells[rng.permutation(nc)]
    cen = coords[cells].mean(axis=1)
    key = cen[:, 0] + 0.7 * cen[:, 1] + 0.4 * cen[:, 2]        # equal slabs along a skew direction
    owner = (np.argsort(np.argsort(key)) * nranks // nc).astype(np.int32)
    return cells, owner, coords


@pytest.mark.parametrize("nranks", [1, 2, 4])
def test_q2_ghost_layer_matches_structured_builder(nranks):
    from pmg_dolfinx_b200 import api
    q = cr.q2_box(3, 3, 2, cr.sector, perturb=0.2)
    cells, owner, coords = scrambled_q2(q, 3, nranks)
    if nranks > 1:
        assert len(np.unique(owner)) == nranks
    meshes = [api.GhostLayerMesh(cells, owner, coords, r, nranks) for r in range(nranks)]
    ctree = cKDTree(q.verts[q.geom_dofmap].mean(axis=1))
    for P in (1, 3):
        Xs = cr.dof_coords(q, P)
        tree = cKDTree(Xs)
        Gs, _ = cr.geometry_factors(q.verts, q.geom_dofmap, P)
        seen = np.zeros(len(Xs), dtype=int)
        for gm in meshes:
            assert gm.nodes_per_cell == 27 and gm.geom_dofmap.shape == (gm.n_cells, 27)
            # the builder carries every cell's 27 nodes as given (rotations included)
            assert np.array_equal(gm.xgeom[gm.geom_dofmap], coords[cells[gm.cell_gid]])
            sp = gm.space(P)
            dist, idx = tree.query(sp.coords)
            assert dist.max() < 1e-12                        # dof coordinates through the quadratic map
            assert len(np.unique(idx)) == len(idx)
            assert np.array_equal(sp.bc, om.bc_marker(q, P)[idx])
            seen[idx[: sp.n_owned]] += 1
            assert sp.n_global == len(Xs)
            # per-rank geometry: each local cell's G is the structured cell's G in a rotated frame, at permuted
            # points -- compare the rotation invariant trace G per cell, as a sorted set over the points
            Gl, detJ = cr.geometry_factors(gm.xgeom, gm.geom_dofmap, P)
            assert (detJ > 0).all()
            sc = ctree.query(gm.xgeom[gm.geom_dofmap].mean(axis=1))[1]
            tr = lambda G: np.sort(G[..., 0] + G[..., 3] + G[..., 5], axis=1)
            assert np.abs(tr(Gl) - tr(Gs[sc])).max() <= 1e-12 * np.abs(tr(Gs)).max()
        assert (seen == 1).all()
    for gm in meshes:
        gm.close()


def test_q2_ghostmesh_rejects_bad_input():
    from pmg_dolfinx_b200.capi import lib, ptr
    q = cr.q2_box(1, 1, 1)
    cells = q.geom_dofmap.astype(np.int64)
    owner = np.zeros(1, dtype=np.int32)
    h = ctypes.c_void_p()
    n = len(q.verts)
    assert lib.pmgx_ghostmesh_create_q2(0, 1, 1, ptr(cells), ptr(owner), n, ptr(q.verts), ctypes.addressof(h)) == 0
    assert lib.pmgx_ghostmesh_nodes_per_cell(h) == 27
    lib.pmgx_ghostmesh_destroy(h)
    bad = cells.copy()
    bad[0, 13] = n                                           # node id out of range
    assert lib.pmgx_ghostmesh_create_q2(0, 1, 1, ptr(bad), ptr(owner), n, ptr(q.verts), ctypes.addressof(h)) != 0
    bad = cells.copy()
    bad[0, 26] = bad[0, 0]                                   # a corner repeated within the cell
    assert lib.pmgx_ghostmesh_create_q2(0, 1, 1, ptr(bad), ptr(owner), n, ptr(q.verts), ctypes.addressof(h)) != 0
    assert b"repeats corner" in lib.pmgx_last_error_string()
