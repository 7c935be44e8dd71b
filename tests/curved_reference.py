"""CPU reference for second-order (27-node) hexahedral geometry, on top of the oracle.

TEST INFRASTRUCTURE ONLY.  The oracle's operator, diagonal, CSR and transfers consume G and dofmaps only; what
changes with a triquadratic map is how G, det J and the dof coordinates come from the nodes, restated here in
numpy:
  * node k = 9a + 3b + c, (a, b, c) in {0, 1, 2}^3 at reference coordinates {0, 1/2, 1} (PMGX_LAP_GEOM_Q2);
  * a Q2 box: the (2n+1)^3 node lattice of the unit cube sent through a map phi, cell (cx, cy, cz) holding
    lattice nodes (2cx + a, 2cy + b, 2cz + c); the dofmap, BC marker and dof count are the oracle's box ones;
  * G = w K K^T / det J and det J at the GLL points, the collocated RHS with lifting, and dof coordinates through
    the quadratic interpolant.
"""
from dataclasses import dataclass

import numpy as np

from oracle import gll, mesh as om, operator as oo

CORNERS = np.array([0, 2, 6, 8, 18, 20, 24, 26])   # corner node of trilinear vertex 4a + 2b + c


@dataclass
class Q2Mesh:
    n: tuple                      # cells per direction
    verts: np.ndarray             # [n_nodes, 3]
    geom_dofmap: np.ndarray       # [nc, 27] int32

    @property
    def ncells(self):
        return int(np.prod(self.n))

    def corners(self):
        """The trilinear mesh on the same corner nodes (an oracle BoxMesh: every oracle function takes it)."""
        return om.BoxMesh(self.n, self.verts, np.ascontiguousarray(self.geom_dofmap[:, CORNERS]))


def sector(X):
    """The annular sector r in [1, 2], theta in [0, pi/2], z in [0, 1] over the unit cube (volume 3 pi / 4)."""
    r, t = 1.0 + X[:, 0], 0.5 * np.pi * X[:, 1]
    return np.stack([r * np.cos(t), r * np.sin(t), X[:, 2]], axis=-1)


def identity(X):
    return X.copy()


def q2_box(nx, ny, nz, phi=identity, perturb=0.0, seed=7):
    """Q2 box through phi; perturb > 0 moves every non-corner node (mid-edge, mid-face, centre) by a seeded
    U(-perturb h/2, perturb h/2)^3, h the cell size of the unit cube."""
    N = (2 * nx + 1, 2 * ny + 1, 2 * nz + 1)
    gx, gy, gz = np.meshgrid(*(np.arange(k) for k in N), indexing="ij")
    X = np.stack([gx / (2 * nx), gy / (2 * ny), gz / (2 * nz)], axis=-1).reshape(-1, 3)
    verts = phi(X)
    if perturb > 0.0:
        mid = ((gx % 2) | (gy % 2) | (gz % 2)).reshape(-1) != 0
        h = np.array([1.0 / nx, 1.0 / ny, 1.0 / nz])
        d = np.random.default_rng(seed).uniform(-0.5 * perturb, 0.5 * perturb, size=verts.shape) * h
        verts[mid] += d[mid]
    cx, cy, cz = (a.reshape(-1) for a in np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij"))
    gd = np.empty((nx * ny * nz, 27), dtype=np.int32)
    for a in range(3):
        for b in range(3):
            for c in range(3):
                gd[:, 9 * a + 3 * b + c] = ((2 * cx + a) * N[1] + (2 * cy + b)) * N[2] + (2 * cz + c)
    return Q2Mesh((nx, ny, nz), verts, gd)


def q2_from_q1(m):
    """The 27-node form of an oracle box whose extra nodes sit at the trilinear positions (the same map)."""
    nx, ny, nz = m.n
    q = q2_box(nx, ny, nz)
    t = np.array([0.0, 0.5, 1.0])
    verts = np.zeros_like(q.verts)
    cv = m.verts[m.geom_dofmap]                                   # [nc, 8, 3]
    for a in range(3):
        for b in range(3):
            for c in range(3):
                w = np.array([(t[a] if i else 1 - t[a]) * (t[b] if j else 1 - t[b]) * (t[c] if k else 1 - t[c])
                              for i in range(2) for j in range(2) for k in range(2)])
                verts[q.geom_dofmap[:, 9 * a + 3 * b + c]] = np.einsum("k,ckd->cd", w, cv)
    return Q2Mesh(m.n, verts, q.geom_dofmap)


def _basis(t):
    """Quadratic Lagrange basis on {0, 1/2, 1} and its derivative, [len(t), 3] each."""
    t = np.asarray(t)[:, None]
    L = np.concatenate([(2 * t - 1) * (t - 1), 4 * t * (1 - t), t * (2 * t - 1)], axis=1)
    D = np.concatenate([4 * t - 3, 4 - 8 * t, 4 * t - 1], axis=1)
    return L, D


def _tensor(P):
    """phi[q, k] and dphi[d, q, k] of the 27 nodes at the (P+1)^3 GLL points, q = ix n^2 + iy n + iz."""
    x1, _ = gll.gll_points_weights(P + 1)
    L, D = _basis(x1)
    phi = np.einsum("ia,jb,kc->ijkabc", L, L, L).reshape(len(x1) ** 3, 27)
    dphi = np.stack([np.einsum("ia,jb,kc->ijkabc", D, L, L), np.einsum("ia,jb,kc->ijkabc", L, D, L),
                     np.einsum("ia,jb,kc->ijkabc", L, L, D)]).reshape(3, len(x1) ** 3, 27)
    return phi, dphi


def geometry_factors(verts, geom_dofmap, P, literal_detj=False):
    """G[c, q, 6] and detJ[c, q] of oracle.operator.geometry_factors for 27-node cells."""
    _, dphi = _tensor(P)
    J = np.einsum("cki,jqk->cqij", verts[geom_dofmap], dphi)
    K = np.empty_like(J)
    K[..., 0, 0] = J[..., 1, 1] * J[..., 2, 2] - J[..., 1, 2] * J[..., 2, 1]
    K[..., 0, 1] = -J[..., 0, 1] * J[..., 2, 2] + J[..., 0, 2] * J[..., 2, 1]
    K[..., 0, 2] = J[..., 0, 1] * J[..., 1, 2] - J[..., 0, 2] * J[..., 1, 1]
    K[..., 1, 0] = -J[..., 1, 0] * J[..., 2, 2] + J[..., 1, 2] * J[..., 2, 0]
    K[..., 1, 1] = J[..., 0, 0] * J[..., 2, 2] - J[..., 0, 2] * J[..., 2, 0]
    K[..., 1, 2] = -J[..., 0, 0] * J[..., 1, 2] + J[..., 0, 2] * J[..., 1, 0]
    K[..., 2, 0] = J[..., 1, 0] * J[..., 2, 1] - J[..., 1, 1] * J[..., 2, 0]
    K[..., 2, 1] = -J[..., 0, 0] * J[..., 2, 1] + J[..., 0, 1] * J[..., 2, 0]
    K[..., 2, 2] = J[..., 0, 0] * J[..., 1, 1] - J[..., 0, 1] * J[..., 1, 0]
    if literal_detj:
        detJ = J[..., 0, 0] * K[..., 0, 0] - J[..., 1, 0] * K[..., 0, 1] + J[..., 0, 2] * K[..., 2, 0]
    else:
        detJ = J[..., 0, 0] * K[..., 0, 0] + J[..., 0, 1] * K[..., 1, 0] + J[..., 0, 2] * K[..., 2, 0]
    KKt = np.einsum("cqik,cqjk->cqij", K, K)
    s = oo.weights_3d(P)[None, :] / detJ
    G = np.stack([KKt[..., 0, 0], KKt[..., 1, 0], KKt[..., 2, 0],
                  KKt[..., 1, 1], KKt[..., 2, 1], KKt[..., 2, 2]], axis=-1) * s[..., None]
    return G, detJ


def dof_coords(mesh, P):
    """Dof coordinates through the triquadratic map."""
    phi, _ = _tensor(P)
    X = np.zeros((om.num_dofs(mesh, P), 3))
    X[om.dofmap(mesh, P).reshape(-1)] = np.einsum("qk,ckd->cqd", phi, mesh.verts[mesh.geom_dofmap]).reshape(-1, 3)
    return X


def rhs_collocated(mesh, P, f, bc, g=0.0, kappa=2.0):
    """oracle.operator.rhs_collocated for 27-node cells: b_i = sum_K f(x_i) w_i |detJ_K(x_i)|, the lifting
    b -= A_full g_bc, then b = g on the BC dofs; f and g are functions of the dof coordinates (or g a scalar)."""
    dm = om.dofmap(mesh, P)
    X = dof_coords(mesh, P)
    G, detJ = geometry_factors(mesh.verts, mesh.geom_dofmap, P)
    b = np.zeros(X.shape[0])
    np.add.at(b, dm.reshape(-1), (f(X)[dm] * (oo.weights_3d(P)[None, :] * np.abs(detJ))).reshape(-1))
    gv = np.full(X.shape[0], float(g)) if np.isscalar(g) else np.asarray(g(X) if callable(g) else g, dtype=np.float64)
    if np.any(gv[bc != 0] != 0.0):
        kap = np.full(mesh.ncells, kappa) if np.isscalar(kappa) else np.asarray(kappa, dtype=np.float64)
        b -= oo.apply(P, dm, G, kap, np.zeros_like(bc), np.where(bc != 0, gv, 0.0))
    b[bc != 0] = gv[bc != 0]
    return b


class Q2Level:
    """tests.helpers.OracleLevel for a 27-node (or, through mesh.corners(), the trilinear) mesh."""

    def __init__(self, mesh, P, kappa=2.0, literal_detj=False):
        self.mesh, self.P = mesh, P
        self.dm = om.dofmap(mesh, P)
        self.bc = om.bc_marker(mesh, P)
        self.nd = om.num_dofs(mesh, P)
        self.kappa = np.full(mesh.ncells, kappa) if np.isscalar(kappa) else np.ascontiguousarray(kappa, dtype=np.float64)
        if mesh.geom_dofmap.shape[1] == 27:
            self.G, self.detJ = geometry_factors(mesh.verts, mesh.geom_dofmap, P, literal_detj)
        else:
            self.G, self.detJ = oo.geometry_factors(mesh.verts, mesh.geom_dofmap, P, literal_detj=literal_detj)

    def A(self, x):
        return oo.apply(self.P, self.dm, self.G, self.kappa, self.bc, x)

    def diag(self):
        return oo.diagonal(self.P, self.dm, self.G, self.kappa, self.bc, self.nd)

    def csr(self):
        return oo.assemble_csr(self.P, self.dm, self.G, self.kappa, self.bc, self.nd)


# the manufactured solution on the sector: zero on its whole boundary
def u_exact(X):
    r, t = np.hypot(X[:, 0], X[:, 1]), np.arctan2(X[:, 1], X[:, 0])
    return np.sin(np.pi * (r - 1)) * np.sin(2 * t) * np.sin(np.pi * X[:, 2])


def f_exact(kappa):
    """-kappa Laplace(u_exact), in cylindrical coordinates."""
    def f(X):
        r, t = np.hypot(X[:, 0], X[:, 1]), np.arctan2(X[:, 1], X[:, 0])
        R, dR = np.sin(np.pi * (r - 1)), np.pi * np.cos(np.pi * (r - 1))
        lap = (-2 * np.pi ** 2 * R + dR / r - 4 * R / r ** 2) * np.sin(2 * t) * np.sin(np.pi * X[:, 2])
        return -kappa * lap
    return f


def volume(mesh, P=4):
    """Sum of the collocated load vector for f = 1 with no BC rows: the quadrature of the mapped domain's volume."""
    ones = lambda X: np.ones(len(X))
    nobc = np.zeros(om.num_dofs(mesh, P), dtype=np.int8)
    if mesh.geom_dofmap.shape[1] == 27:
        return rhs_collocated(mesh, P, ones, nobc).sum()
    return oo.rhs_collocated(mesh, P, ones, nobc).sum()


def coords_of(mesh, P):
    return dof_coords(mesh, P) if mesh.geom_dofmap.shape[1] == 27 else om.dof_coords(mesh, P)


def nodal_error(mesh, P=4, kappa=1.0):
    """max |u_h - u| / max |u| at the dofs, u_h the direct solve of the collocated system."""
    import scipy.sparse.linalg as spla
    lv = Q2Level(mesh, P, kappa)
    X = coords_of(mesh, P)
    if mesh.geom_dofmap.shape[1] == 27:
        b = rhs_collocated(mesh, P, f_exact(kappa), lv.bc)
    else:
        b = oo.rhs_collocated(mesh, P, f_exact(kappa), lv.bc)
    uh = spla.spsolve(lv.csr().tocsc(), b)
    u = u_exact(X)
    return np.abs(uh - u).max() / np.abs(u).max()
