"""GPU parity of the p-transfers for every degree pair 1 <= Pc <= Pf <= 8.

interp.cu instantiates k_prolong / k_restrict for every pair, each with its own threads per CTA and cells per CTA
(XferCfg).  Here each pair runs on a general mesh from the ghost-layer builder: the box of test_ghostmesh.py's
scrambled_box, with randomly numbered vertices and cells and every cell's local frame rotated, so neighbouring cells
see their shared dofs in different orientations.  The cell list is permuted and split raggedly into lcells and
bcells.  Prolongation and restriction are compared with the oracle on the builder's dofmaps, R = P^T is checked,
and on the unperturbed mesh prolongation must reproduce a tensor polynomial of the coarse degree exactly.

The fused forms of the V-cycle (prolongation that adds into u, restriction of fine - sub) only run inside a cycle:
three-level chains that no other test runs are compared stage by stage with the oracle's V-cycle.
"""
import numpy as np
import pytest

from oracle import mesh as om, operator as oo, solvers as osol
from test_ghostmesh import scrambled_box
from test_gpu_solvers import _build_hierarchy

pytestmark = pytest.mark.gpu
PAIRS = [(pc, pf) for pf in range(1, 9) for pc in range(1, pf + 1)]
BOX = (5, 5, 4)  # 100 cells: even the (1, 1) pair, 64 cells per CTA, has CTAs of more than one cell in both lists


@pytest.fixture(scope="module")
def general_meshes():
    from pmg_dolfinx_b200 import api
    out = {}
    for perturb in (0.0, 0.15):
        _, cells, owner, coords = scrambled_box(BOX, perturb, 17, 1)
        gm = api.GhostLayerMesh(cells, owner, coords, 0, 1)
        out[perturb] = (gm, {P: gm.space(P) for P in range(1, 9)})
    yield out
    for gm, _ in out.values():
        gm.close()


@pytest.mark.parametrize("perturb", [0.0, 0.15])
@pytest.mark.parametrize("Pc,Pf", PAIRS)
def test_prolong_restrict_pair_on_a_general_mesh(ctx, general_meshes, Pc, Pf, perturb):
    from pmg_dolfinx_b200 import api
    gm, spaces = general_meshes[perturb]
    sc, sf = spaces[Pc], spaces[Pf]
    assert sc.n_ghost == 0 and sf.n_ghost == 0
    nc, nf = sc.n_owned, sf.n_owned
    rng = np.random.default_rng(100 * Pc + 10 * Pf + int(perturb > 0))
    perm = rng.permutation(gm.n_cells).astype(np.int32)
    split = 59  # 59 and 41 cells: ragged against every cells-per-CTA count of XferCfg (128 / 64 / 32 threads over Pf + 1)
    dmc, dmf = ctx.to_device(sc.dofmap), ctx.to_device(sf.dofmap)
    it = api.Interpolator(ctx, Pc, Pf, dmc, dmf, nc, nf, perm[:split], perm[split:])
    vc, vf = api.Vector(ctx, nc), api.Vector(ctx, nf)

    xc = rng.uniform(-1, 1, nc)
    vc.copy_from_host(xc)
    vf.set(-7.5e30)  # the output is overwritten
    it.interpolate(vc, vf)
    po = oo.prolong(Pc, Pf, sc.dofmap, sf.dofmap, xc, nf)
    pf_ = vf.data_copy()
    assert np.abs(pf_ - po).max() / np.abs(po).max() < 1e-13, (Pc, Pf, perturb)

    xf = rng.uniform(-1, 1, nf)
    vf.copy_from_host(xf)
    vc.set(123.0)  # the output is zeroed first (interpolate.hpp:270)
    it.reverse_interpolate(vf, vc)
    ro = oo.restrict(Pc, Pf, sc.dofmap, sf.dofmap, xf, nc)   # multiplicity over all cells
    rg = vc.data_copy()
    assert np.abs(rg - ro).max() / np.abs(ro).max() < 1e-13, (Pc, Pf, perturb)

    # R = P^T: (P u_c, w) = (u_c, R w)
    a, b = np.dot(pf_, xf), np.dot(xc, rg)
    assert abs(a - b) <= 1e-12 * np.linalg.norm(pf_) * np.linalg.norm(xf), (a, b)

    if perturb == 0.0:
        # known answer: every cell is an axis-aligned box, so a product of 1-D polynomials of degree Pc is in the
        # coarse space and the prolongation reproduces it at the fine dofs
        coef = rng.uniform(-1, 1, (3, Pc + 1))
        poly = lambda X: np.prod([np.polynomial.polynomial.polyval(X[:, d], coef[d]) for d in range(3)], axis=0)
        vc.copy_from_host(poly(sc.coords[:nc]))
        vf.set(-7.5e30)
        it.interpolate(vc, vf)
        exact = poly(sf.coords[:nf])
        assert np.abs(vf.data_copy() - exact).max() <= 1e-12 * np.abs(exact).max(), (Pc, Pf)


@pytest.mark.parametrize("degrees", [(1, 4, 8), (2, 5, 7), (3, 6, 8)])
def test_vcycle_fused_transfers_on_new_chains(ctx, degrees):
    """Four V-cycles: with per-stage diagnostics (flags 2: the prolongation adds into u in its store) the stage
    residual norms of test_vcycle_history against the oracle, and in the production cycle (flags 0: the restriction
    also takes fine - sub, sub the last r -= q of the smoother) the iterates."""
    from pmg_dolfinx_b200 import api
    mesh = om.create_box(3, 2, 2, perturb=0.1)
    ols, gls, olev, smoothers, interps, pro, res = _build_hierarchy(ctx, mesh, degrees)
    top = ols[-1]
    b = oo.rhs_collocated(mesh, top.P, oo.f_sines(1, 1, 1, 2.0), top.bc)
    for flags in (2, 0):
        pmg = api.MultigridPreconditioner(ctx, [g.bc for g in gls], flags=flags)
        pmg.set_solvers(smoothers)
        pmg.set_operators([g.op for g in gls])
        pmg.set_interpolators(interps)
        pmg.set_coarse_solver(None)
        u, bv = gls[-1].vec(), gls[-1].vec(b)
        uo = np.zeros(top.nd)
        for it in range(4):
            ho = []
            uo = osol.vcycle(olev, pro, res, b, uo, history=ho)
            rn = pmg.apply(bv, u, verbose=True)
            hov = np.array([h[2] for h in ho])
            if flags == 2:
                hg = pmg.diagnostics()
                assert len(hg) == len(hov)
                assert np.all(np.abs(hg - hov) <= 1e-9 * hov[0]), (degrees, it, hg, hov)
            assert abs(rn - hov[-1]) <= 1e-9 * hov[0], (degrees, flags, it)
            ur = u.data_copy()
            assert np.linalg.norm(ur - uo) <= 1e-9 * np.linalg.norm(uo), (degrees, flags, it)
