"""GPU parity: matrix-free Laplacian, geometry factors, diagonal (SURVEY 8 rows a1-a4).

Tolerance (north_star): operator action relative 1e-12 in FP64, max- and 2-norm, against the
oracle on the same mesh, degree and input; checked on the uniform cube and on the seeded
perturbed mesh (which exposes G-indexing errors the uniform cube hides, quirk Q1).
"""
import numpy as np
import pytest

from oracle import mesh as om, operator as oo
from helpers import OracleLevel, GpuLevel, rel

pytestmark = pytest.mark.gpu
TOL = 1e-12

# The apply kernel of every degree, as kernel_name() reports it: (every cell affine, G streamed per quadrature point)
KERNELS = {
    1: ("k_apply_affine<1,128>", "k_apply_tma<1,64,2>"),
    2: ("k_apply_affine_shfl<2,128>", "k_apply_tma<2,128,2>"),
    3: ("k_apply_affine2<3,64,warp-local>", "k_apply_tma<3,128,2>"),
    4: ("k_apply_affine<4,64>", "k_apply_tma<4,128,2>"),
    5: ("k_apply_affine<5,64>", "k_apply_tma<5,64,2>"),
    6: ("k_apply_affine_mma<6,2,affine>", "k_apply_affine_mma<6,2,streamed>"),
    7: ("k_apply_affine_mma<7,2,affine>", "k_apply_affine_mma<7,2,streamed>"),
    8: ("k_apply<8>", "k_apply<8>"),
}


@pytest.mark.parametrize("P", [1, 2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("perturb", [0.0, 0.2])
def test_apply_matches_oracle(ctx, P, perturb):
    """Both apply kernels of every degree: the uniform box takes the affine one (except at P8, which has none),
    the perturbed box and PMGX_LAP_STREAM_G (flags=4) on the uniform box the streamed-G one."""
    n = (3, 4, 5) if P <= 4 else (2, 3, 2)
    ol = OracleLevel(om.create_box(*n, perturb=perturb), P)
    levels = [(GpuLevel(ctx, ol), KERNELS[P][0 if perturb == 0.0 else 1])]
    if perturb == 0.0:
        levels.append((GpuLevel(ctx, ol, flags=4), KERNELS[P][1]))
    rng = np.random.default_rng(42)
    for gl, kernel in levels:
        assert gl.op.kernel_name() == kernel, (P, perturb, gl.op.kernel_name())
        assert gl.op.is_affine() == (kernel == KERNELS[P][0] and P != 8)
        for x in (rng.uniform(-1, 1, ol.nd), np.ones(ol.nd)):
            y, yo = gl.apply(x), ol.A(x)
            e2, einf = rel(y, yo)
            assert e2 < TOL and einf < TOL, (P, perturb, kernel, e2, einf)


@pytest.mark.parametrize("P", [1, 3, 4, 6])
def test_apply_cell_lists_and_ragged_batches(ctx, P):
    """lcells/bcells in arbitrary order, sizes not a multiple of the cells-per-block batch."""
    ol = OracleLevel(om.create_box(3, 3, 5, perturb=0.15), P)
    rng = np.random.default_rng(7)
    perm = rng.permutation(ol.mesh.ncells).astype(np.int32)
    gl = GpuLevel(ctx, ol, lcells=perm[:17], bcells=perm[17:])
    x = rng.uniform(-1, 1, ol.nd)
    e2, einf = rel(gl.apply(x), ol.A(x))
    assert e2 < TOL and einf < TOL


def test_apply_subset_of_cells_and_empty_lists(ctx):
    """Only the listed cells contribute (reference: entities list, laplacian.hpp:182); empty
    lists give y = 0."""
    P = 2
    ol = OracleLevel(om.create_box(3, 3, 3), P)
    cells = np.array([0, 5, 13, 26], dtype=np.int32)
    gl = GpuLevel(ctx, ol, lcells=cells[:1], bcells=cells[1:])
    x = np.random.default_rng(3).uniform(-1, 1, ol.nd)
    yo = oo.apply_cells(P, ol.dm, ol.G, ol.kappa, ol.bc, x, np.zeros(ol.nd), cells)
    e2, _ = rel(gl.apply(x), yo)
    assert e2 < TOL
    g0 = GpuLevel(ctx, ol, lcells=np.zeros(0, np.int32), bcells=np.zeros(0, np.int32))
    assert np.abs(g0.apply(x)).max() == 0.0


@pytest.mark.parametrize("P", [1, 2, 3, 4, 6])
def test_geometry_factors_match_oracle(ctx, P):
    for literal in (False, True):
        ol = OracleLevel(om.create_box(2, 3, 2, perturb=0.2), P, literal_detj=literal)
        gl = GpuLevel(ctx, ol, flags=1 if literal else 0)
        G = gl.op.geometry_factors()
        assert np.abs(G - ol.G).max() / np.abs(ol.G).max() < 1e-13


def test_uniform_cube_G_is_diagonal(ctx):
    """Known answer (SURVEY 8c): uniform cube with h = 1/n gives G = diag(h w_q)."""
    n, P = 4, 3
    ol = OracleLevel(om.create_box(n, n, n), P)
    G = GpuLevel(ctx, ol).op.geometry_factors()
    w = oo.weights_3d(P)
    assert np.abs(G[:, :, [1, 2, 4]]).max() < 1e-15 * np.abs(G).max()
    for c in (0, 3, 5):
        assert np.allclose(G[:, :, c], w[None, :] / n, rtol=1e-14, atol=0)


@pytest.mark.parametrize("P", [1, 2, 3, 4, 5, 6, 7, 8])
def test_diag_inverse_matches_assembled_diagonal(ctx, P):
    n = (3, 2, 3) if P <= 4 else (2, 2, 2)
    ol = OracleLevel(om.create_box(*n, perturb=0.2), P)
    gl = GpuLevel(ctx, ol)
    v = gl.vec()
    gl.op.get_diag_inverse(v)
    d = 1.0 / v.data_copy()
    do = ol.diag()
    assert np.abs(d - do).max() / np.abs(do).max() < 1e-13
    assert (d[ol.bc != 0] == 1.0).all()


def test_known_answers_constant_and_linear(ctx):
    """A * const = 0 and A * linear = 0 at rows whose cells touch no Dirichlet dof (affine mesh)."""
    P, n = 3, 4
    ol = OracleLevel(om.create_box(n, n, n), P)
    gl = GpuLevel(ctx, ol)
    X = om.dof_coords(ol.mesh, P)
    touched = np.zeros(ol.nd, dtype=bool)
    cell_has_bc = (ol.bc[ol.dm] != 0).any(axis=1)
    touched[ol.dm[cell_has_bc].reshape(-1)] = True
    scale = np.abs(ol.A(np.random.default_rng(0).uniform(-1, 1, ol.nd))).max()
    for f in (np.ones(ol.nd), X[:, 0] + 2 * X[:, 1] - X[:, 2]):
        y = gl.apply(f)
        assert np.abs(y[~touched]).max() < 1e-13 * scale


def test_symmetry(ctx):
    ol = OracleLevel(om.create_box(3, 3, 3, perturb=0.2), 4)
    gl = GpuLevel(ctx, ol)
    rng = np.random.default_rng(5)
    x, y = rng.uniform(-1, 1, ol.nd), rng.uniform(-1, 1, ol.nd)
    x[ol.bc != 0] = 0
    y[ol.bc != 0] = 0
    a, b = np.dot(y, gl.apply(x)), np.dot(x, gl.apply(y))
    assert abs(a - b) < 1e-12 * abs(a)


def test_unsupported_degree_and_size_errors(ctx):
    from pmg_dolfinx_b200 import api
    ol = OracleLevel(om.create_box(2, 2, 2), 2)
    gl = GpuLevel(ctx, ol)
    with pytest.raises(api.PmgxError, match="Unsupported degree"):
        api.MatFreeLaplacian(ctx, 9, gl.kappa, gl.dofmap, gl.xgeom, gl.gdm, gl.lcells, gl.bcells, gl.bc, ol.nd)
    with pytest.raises(api.PmgxError):
        api.MatFreeLaplacian(ctx, 2, gl.kappa, gl.dofmap, gl.xgeom, gl.gdm, np.array([99], np.int32), gl.bcells,
                             gl.bc, ol.nd)
    a, b = api.Vector(ctx, 5), api.Vector(ctx, 6)
    with pytest.raises(api.PmgxError, match="Incompatible vector sizes"):
        api.inner_product(a, b)


@pytest.mark.parametrize("P", [1, 2, 3, 4, 5, 6])
def test_affine_geometry_kernel_on_a_sheared_box(ctx, P):
    """Every cell of a linearly mapped box is a parallelepiped: the operator takes the affine-geometry
    kernel (one geometry 6-vector per cell, G(q) = w_q Gc with all six components non-zero) and must
    give the oracle's action, the streamed-G kernel's action (PMGX_LAP_STREAM_G) and the same
    diagonal; a single displaced vertex sends the operator back to the streamed kernels."""
    mesh = om.create_box(4, 3, 5)
    M = np.array([[1.0, 0.3, -0.2], [0.1, 0.9, 0.25], [-0.15, 0.2, 1.1]])
    mesh.verts[:] = mesh.verts @ M.T + np.array([0.3, -1.0, 2.0])
    ol = OracleLevel(mesh, P)
    assert np.abs(ol.G[:, :, [1, 2, 4]]).max() > 1e-3          # genuinely non-diagonal geometry
    gl, gs = GpuLevel(ctx, ol), GpuLevel(ctx, ol, flags=4)
    assert gl.op.is_affine() and not gs.op.is_affine()
    x = np.random.default_rng(P).uniform(-1, 1, ol.nd)
    ya, ys, yo = gl.apply(x), gs.apply(x), ol.A(x)
    assert rel(ya, yo)[1] < 1e-12 and rel(ys, yo)[1] < 1e-12 and rel(ya, ys)[1] < 1e-13
    # ragged batches / split lists through the affine kernel
    nc = mesh.ncells
    cells = np.arange(nc, dtype=np.int32)
    g2 = GpuLevel(ctx, ol, lcells=cells[: nc // 3], bcells=cells[nc // 3:])
    assert g2.op.is_affine() and rel(g2.apply(x), yo)[1] < 1e-12
    # one displaced vertex: not affine any more, still correct
    mesh2 = om.create_box(4, 3, 5)
    mesh2.verts[:] = mesh2.verts @ M.T
    mesh2.verts[37] += 1e-6
    ol2 = OracleLevel(mesh2, P)
    gl2 = GpuLevel(ctx, ol2)
    assert not gl2.op.is_affine()
    assert rel(gl2.apply(x), ol2.A(x))[1] < 1e-12


@pytest.mark.parametrize("P,perturb", [(1, 0.0), (3, 0.2), (4, 0.0), (6, 0.15)])
def test_rhs_with_lifting_matches_oracle_and_reproduces_constants(ctx, P, perturb):
    """assemble_vector + apply_lifting + set_bc with inhomogeneous Dirichlet data g = 1.3
    (examples/cg/main.cpp:158,234-236; examples/pmg/main.cpp:293-295): b equals the oracle's, and the
    known answer -- with f = 0 the solution of A u = b is the constant g (constants are in the kernel of
    the unconstrained operator) -- comes out of a CG solve."""
    from pmg_dolfinx_b200 import api
    import torch
    mesh = om.create_box(4, 3, 5, perturb=perturb)
    ol = OracleLevel(mesh, P, kappa=np.random.default_rng(3).uniform(0.5, 2.0, mesh.ncells))
    gl = GpuLevel(ctx, ol)
    X = om.dof_coords(mesh, P)
    f = lambda Y: 1000.0 * np.exp(-((Y[:, 0] - 0.5) ** 2 + (Y[:, 1] - 0.5) ** 2) / 0.02)   # examples/cg/main.cpp:136-148
    g = 1.3
    bo = oo.rhs_collocated(mesh, P, f, ol.bc, g=g, kappa=ol.kappa)
    bv = gl.vec()
    gl.op.assemble_rhs(ctx.to_device(f(X)), g, bv)
    assert rel(bv.data_copy(), bo)[0] < 1e-12
    # lifting really changed the free rows next to the boundary
    b0 = oo.rhs_collocated(mesh, P, f, ol.bc, g=0.0)
    free = ol.bc == 0
    assert np.linalg.norm((bo - b0)[free]) > 1e-3 * np.linalg.norm(b0[free])
    # per-dof Dirichlet data through the vector entry point
    gvec = np.where(ol.bc != 0, 1.0 + X[:, 0] - 2.0 * X[:, 2], 7.0)
    bo2 = oo.rhs_collocated(mesh, P, f, ol.bc, g=gvec, kappa=ol.kappa)
    bv2 = gl.vec()
    gl.op.assemble_rhs(ctx.to_device(f(X)), 0.0, bv2)
    gl.op.lift(ctx.to_device(gvec), bv2)
    assert rel(bv2.data_copy(), bo2)[0] < 1e-12
    # known answer: f = 0, g constant -> u = g
    bz = gl.vec()
    gl.op.assemble_rhs(ctx.to_device(np.zeros(ol.nd)), g, bz)
    cg = api.CGSolver(ctx, ol.nd, 0)
    cg.set_max_iterations(400)
    cg.set_tolerance(1e-12)
    u = gl.vec()
    cg.solve(gl.op, u, bz)
    assert np.abs(u.data_copy() - g).max() < 1e-8
