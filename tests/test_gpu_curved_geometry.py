"""GPU: second-order (27-node) geometry, PMGX_LAP_GEOM_Q2, against the CPU reference of tests/curved_reference.py
on the annular sector with its mid-edge, mid-face and centre nodes perturbed: G, apply, diagonal, CSR, RHS and
lifting at P1..P8; the reduction to the 8-node operator; a P4 -> P2 -> P1 multigrid-preconditioned CG solve; the
convergence orders of tests/test_curved_geometry_cpu.py; and a scrambled general 27-node mesh through the
ghost-layer builder."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla
from scipy.spatial import cKDTree

from oracle import mesh as om, operator as oo, solvers as osol
from helpers import GpuLevel, OracleLevel, rel
import curved_reference as cr
from test_curved_geometry_cpu import MIN_GAIN, Q2_MIN_ORDER, scrambled_q2

pytestmark = pytest.mark.gpu


def curved(n=(3, 2, 2)):
    return cr.q2_box(*n, phi=cr.sector, perturb=0.1)


def q2_flags(api, mesh, flags=0):
    return flags | (api.LAP_GEOM_Q2 if mesh.geom_dofmap.shape[1] == 27 else 0)


@pytest.mark.parametrize("P", range(1, 9))
def test_geometry_factors_match_reference(ctx, P):
    """Exact det J on the perturbed sector; LAP_LITERAL_DETJ on a unit box with perturbed mid-edge, mid-face and
    centre nodes.  The reference's literal expression equals det J only near axis-aligned cells: on the sector it
    comes close to zero at some points, and there G itself is ill-conditioned (errors of 1e-11 relative to max |G|
    measured between two correct evaluations), which says nothing about the kernel."""
    from pmg_dolfinx_b200 import api
    for lit in (False, True):
        m = cr.q2_box(3, 2, 2, perturb=0.1) if lit else curved()
        ol = cr.Q2Level(m, P, literal_detj=lit)
        gl = GpuLevel(ctx, ol, flags=api.LAP_GEOM_Q2 | (api.LAP_LITERAL_DETJ if lit else 0))
        assert not gl.op.is_affine()
        G = gl.op.geometry_factors()
        assert np.abs(G - ol.G).max() / np.abs(ol.G).max() < 1e-13


@pytest.mark.parametrize("P", range(1, 9))
def test_operator_matches_reference(ctx, P):
    """apply 1e-12, diagonal 1e-13, assembled CSR, RHS with non-constant Dirichlet data through lift."""
    from pmg_dolfinx_b200 import api
    m = curved()
    kap = 1.0 + np.arange(m.ncells) % 3
    ol = cr.Q2Level(m, P, kappa=kap)
    gl = GpuLevel(ctx, ol, flags=api.LAP_GEOM_Q2)
    x = np.random.default_rng(P).uniform(-1, 1, ol.nd)
    assert rel(gl.apply(x), ol.A(x))[1] < 1e-12
    dinv = gl.vec()
    gl.op.get_diag_inverse(dinv)
    d = 1.0 / dinv.data_copy()
    do = ol.diag()
    assert np.abs(d - do).max() / np.abs(do).max() < 1e-13
    rp, co, va = gl.op.to_csr().to_host()
    A = sp.csr_matrix((va, co, rp), shape=(ol.nd, ol.nd))
    Ao = ol.csr()
    assert abs(A - Ao).max() <= 1e-13 * abs(Ao).max()
    # b = f w |det J| at the dofs, lifted with g(x) on the boundary
    X = cr.dof_coords(m, P)
    f = lambda X: 1.0 + X[:, 0] * X[:, 1]
    g = lambda X: np.sin(X[:, 0]) + X[:, 2] ** 2
    bo = cr.rhs_collocated(m, P, f, ol.bc, g=g, kappa=kap)
    fv, gv = ctx.to_device(f(X)), ctx.to_device(g(X))
    bv = gl.vec()
    gl.op.assemble_rhs(fv, 0.0, bv)
    gl.op.lift(gv, bv)
    assert rel(bv.data_copy(), bo)[0] < 1e-12


@pytest.mark.parametrize("P", [1, 3, 4, 6, 8])
def test_reduction_to_trilinear(ctx, P):
    from pmg_dolfinx_b200 import api
    # the uniform box as a 27-node mesh: affine, the same kernel and apply as the 8-node form
    m = om.create_box(3, 4, 2)
    q = cr.q2_from_q1(m)
    o1, o2 = OracleLevel(m, P), cr.Q2Level(q, P)
    g1, g2 = GpuLevel(ctx, o1), GpuLevel(ctx, o2, flags=api.LAP_GEOM_Q2)
    assert g2.op.is_affine() == g1.op.is_affine() == (P < 8)
    assert g2.op.kernel_name() == g1.op.kernel_name()
    x = np.random.default_rng(1).uniform(-1, 1, o1.nd)
    assert rel(g2.apply(x), g1.apply(x))[0] < 1e-13
    # a perturbed box with its extra nodes at the trilinear positions: the 8-node G, diagonal and CSR
    m = om.create_box(3, 4, 2, perturb=0.2)
    q = cr.q2_from_q1(m)
    g1, g2 = GpuLevel(ctx, OracleLevel(m, P)), GpuLevel(ctx, cr.Q2Level(q, P), flags=api.LAP_GEOM_Q2)
    assert not g2.op.is_affine() and g2.op.kernel_name() == g1.op.kernel_name()
    G1, G2 = g1.op.geometry_factors(), g2.op.geometry_factors()
    assert np.abs(G2 - G1).max() <= 1e-13 * np.abs(G1).max()
    d1, d2 = g1.vec(), g2.vec()
    g1.op.get_diag_inverse(d1)
    g2.op.get_diag_inverse(d2)
    assert rel(d2.data_copy(), d1.data_copy())[1] < 1e-13
    (rp1, co1, va1), (rp2, co2, va2) = g1.op.to_csr().to_host(), g2.op.to_csr().to_host()
    assert np.array_equal(rp1, rp2) and np.array_equal(co1, co2)
    assert np.abs(va2 - va1).max() <= 1e-13 * np.abs(va1).max()


def test_q2_with_recompute_is_unsupported(ctx):
    from pmg_dolfinx_b200 import api
    from pmg_dolfinx_b200.capi import PmgxError
    ol = cr.Q2Level(curved(), 2)
    with pytest.raises(PmgxError) as e:
        GpuLevel(ctx, ol, flags=api.LAP_GEOM_Q2 | api.LAP_RECOMPUTE_G)
    assert e.value.code == 5 and "PMGX_LAP_GEOM_Q2" in e.value.msg


def pmg_solve(ctx, mesh, degrees, kappa, f, rtol=1e-12):
    """P-multigrid-preconditioned CG (Chebyshev smoothers, AMG coarse solve) of the collocated problem."""
    from pmg_dolfinx_b200 import api
    flags = q2_flags(api, mesh)
    ols = [cr.Q2Level(mesh, P, kappa) for P in degrees]
    gls = [GpuLevel(ctx, ol, flags=flags) for ol in ols]
    smoothers = []
    for ol, gl in zip(ols, gls):
        cg = api.CGSolver(ctx, ol.nd, 0)
        cg.set_max_iterations(20)
        cg.set_tolerance(1e-6)
        cg.store_coefficients(True)
        cg.solve(gl.op, gl.vec(), gl.vec(np.ones(ol.nd)))
        lmax = cg.compute_eigenvalues()[-1]
        s = api.Chebyshev(ctx, ol.nd, 0, (0.1 * lmax, 1.1 * lmax))
        s.set_max_iterations(2)
        smoothers.append(s)
    allc = np.arange(mesh.ncells, dtype=np.int32)
    interps = [api.Interpolator(ctx, a.P, b.P, ga.dofmap, gb.dofmap, a.nd, b.nd, allc, allc[:0])
               for a, b, ga, gb in zip(ols[:-1], ols[1:], gls[:-1], gls[1:])]
    cs = api.CoarseSolverType(ctx, gls[0].op.to_csr(), 60, 1e-10, amg=True, min_coarse=100)
    pmg = api.MultigridPreconditioner(ctx, [g.bc for g in gls])
    pmg.set_solvers(smoothers)
    pmg.set_operators([g.op for g in gls])
    pmg.set_interpolators(interps)
    pmg.set_coarse_solver(cs)
    top, gtop = ols[-1], gls[-1]
    b = cr.rhs_collocated(mesh, top.P, f, top.bc) if flags else oo.rhs_collocated(mesh, top.P, f, top.bc)
    cg = api.CGSolver(ctx, top.nd, 0)
    cg.set_max_iterations(100)
    cg.set_tolerance(rtol)
    cg.set_preconditioner(pmg)
    x = gtop.vec()
    its = cg.solve(gtop.op, x, gtop.vec(b))
    return x.data_copy(), b, top, its


def test_pmg_cg_solve_on_the_sector(ctx):
    m = cr.q2_box(4, 4, 4, cr.sector)
    u, b, top, its = pmg_solve(ctx, m, (1, 2, 4), 1.0, cr.f_exact(1.0))
    uo = spla.spsolve(sp.csc_matrix(top.csr()), b)
    assert its < 100 and rel(u, uo)[0] < 1e-8, its


def test_geometry_order_on_gpu(ctx):
    """The GPU's volume and P4 nodal error show the orders the CPU reference calibrated (the nodal error at n = 4
    and 8: at n = 2 the P1 level is too small for the smoothers' eigenvalue estimate)."""
    from pmg_dolfinx_b200 import api

    def volume(mesh, P=4):
        ol = cr.Q2Level(mesh, P)
        ol.bc = np.zeros_like(ol.bc)
        gl = GpuLevel(ctx, ol, flags=q2_flags(api, mesh))
        bv = gl.vec()
        gl.op.assemble_rhs(ctx.to_device(np.ones(ol.nd)), 0.0, bv)
        return bv.data_copy().sum()

    def nodal_error(mesh):
        u, *_ = pmg_solve(ctx, mesh, (1, 2, 4), 1.0, cr.f_exact(1.0))
        ue = cr.u_exact(cr.coords_of(mesh, 4))
        return np.abs(u - ue).max() / np.abs(ue).max()

    exact = 0.75 * np.pi
    for err, ns in ((lambda m: abs(volume(m) - exact), (4, 8)), (nodal_error, (4, 8))):
        q2 = [cr.q2_box(n, n, n, cr.sector) for n in ns]
        e2 = [err(m) for m in q2]
        e1 = [err(m.corners()) for m in q2]
        o2, o1 = np.log2(e2[0] / e2[1]), np.log2(e1[0] / e1[1])
        assert o2 > Q2_MIN_ORDER and o2 > o1 + MIN_GAIN, (e1, e2)


def test_general_q2_mesh_single_gpu(ctx):
    """A renumbered, shuffled and rotated 27-node sector through pmgx_ghostmesh_create_q2 on one rank: apply
    against the structured reference (matched by dof coordinates), and three P4 -> P2 -> P1 V-cycles against the
    oracle's cycle on the same arrays."""
    from pmg_dolfinx_b200 import api
    q = curved((3, 3, 2))
    cells, owner, coords = scrambled_q2(q, 11, 1)
    gm = api.GhostLayerMesh(cells, owner, coords)
    degrees = (1, 2, 4)
    levels = []
    for P in degrees:
        s = gm.space(P)
        idx = cKDTree(cr.dof_coords(q, P)).query(s.coords)[1]
        ol = cr.Q2Level(q, P)                             # structured reference, for the apply
        lv = cr.Q2Level.__new__(cr.Q2Level)              # the general arrays
        lv.mesh, lv.P, lv.dm, lv.bc, lv.nd = gm, P, s.dofmap, s.bc, s.n_owned
        lv.kappa = np.full(gm.n_cells, 2.0)
        lv.G, lv.detJ = cr.geometry_factors(gm.xgeom, gm.geom_dofmap, P)
        g = GpuLevel.__new__(GpuLevel)
        g.ctx, g.ol = ctx, lv
        g.dofmap, g.xgeom, g.gdm = ctx.to_device(s.dofmap), ctx.to_device(gm.xgeom), ctx.to_device(gm.geom_dofmap)
        g.kappa, g.bc = ctx.to_device(lv.kappa), ctx.to_device(s.bc)
        g.op = api.MatFreeLaplacian(ctx, P, g.kappa, g.dofmap, g.xgeom, g.gdm, gm.lcells, gm.bcells, g.bc, s.n_owned,
                                    0, None, api.LAP_GEOM_Q2)
        x = np.random.default_rng(P).uniform(-1, 1, ol.nd)
        assert rel(g.apply(x[idx]), ol.A(x)[idx])[1] < 1e-12
        levels.append((lv, g))
    olev, smoothers, pro, res = [], [], [], []
    for lv, g in levels:
        dinv = 1.0 / lv.diag()
        _, _, al, be, _, _ = osol.cg(lv.A, dinv, np.zeros(lv.nd), np.ones(lv.nd), 20, 1e-6)
        lmax = 1.1 * osol.lanczos_eigenvalues(al, be)[-1]
        olev.append(osol.Level(lv.A, dinv, lv.bc.astype(float), lmax, 2))
        s = api.Chebyshev(ctx, lv.nd, 0, (0.1 * lmax / 1.1, lmax))
        s.set_max_iterations(2)
        smoothers.append(s)
    allc = np.arange(gm.n_cells, dtype=np.int32)
    interps = []
    for (a, ga), (b, gb) in zip(levels[:-1], levels[1:]):
        interps.append(api.Interpolator(ctx, a.P, b.P, ga.dofmap, gb.dofmap, a.nd, b.nd, allc, allc[:0]))
        pro.append((lambda a, b: lambda xc: oo.prolong(a.P, b.P, a.dm, b.dm, xc, b.nd))(a, b))
        res.append((lambda a, b: lambda xf: oo.restrict(a.P, b.P, a.dm, b.dm, xf, a.nd))(a, b))
    c0 = levels[0][0]
    A0 = oo.assemble_csr(c0.P, c0.dm, c0.G, c0.kappa, c0.bc, c0.nd)
    d0 = 1.0 / A0.diagonal()
    cs_o = lambda u0, b0: osol.cg(lambda v: A0 @ v, d0, u0, b0, 60, 1e-10)[0]
    cs_g = api.CoarseSolverType(ctx, levels[0][1].op.to_csr(), 60, 1e-10, amg=True, min_coarse=100)
    pmg = api.MultigridPreconditioner(ctx, [g.bc for _, g in levels], flags=2)
    pmg.set_solvers(smoothers)
    pmg.set_operators([g.op for _, g in levels])
    pmg.set_interpolators(interps)
    pmg.set_coarse_solver(cs_g)
    top, gtop = levels[-1]
    b = np.where(top.bc != 0, 0.0, 1.0)
    u, bv, uo = gtop.vec(), gtop.vec(b), np.zeros(top.nd)
    for _ in range(3):
        uo = osol.vcycle(olev, pro, res, b, uo, coarse_solve=cs_o)
        pmg.apply(bv, u)
        assert rel(u.data_copy(), uo)[0] < 1e-9
    gm.close()
