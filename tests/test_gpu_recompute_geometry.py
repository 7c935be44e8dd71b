"""GPU: the operator that keeps no geometry (PMGX_LAP_RECOMPUTE_G, the reference's batch_size > 0 mode).

Every apply forms G from the mesh inside the kernel, so does every set-up path that reads G (diagonal, CSR
assembly, get_G, lifting).  The results must equal the oracle's and the default operator's to the tolerances
of test_gpu_operator.py, on meshes large enough that every persistent CTA walks over several batches.
"""
import os
import re
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oracle import mesh as om, operator as oo, solvers as osol
from helpers import OracleLevel, GpuLevel, rel

pytestmark = pytest.mark.gpu
TOL = 1e-12
LITERAL, STREAM, RECOMPUTE = 1, 4, 8
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# The recompute kernel of every degree, as kernel_name() reports it
KERNELS = {
    1: "k_apply_tma<1,64,recomputed>",
    2: "k_apply_tma<2,128,recomputed>",
    3: "k_apply_tma<3,128,recomputed>",
    4: "k_apply_tma<4,128,recomputed>",
    5: "k_apply_tma<5,64,recomputed>",
    6: "k_apply_affine_mma<6,2,recomputed>",
    7: "k_apply_affine_mma<7,2,recomputed>",
    8: "k_apply<8,recomputed>",
}


def _mesh(case, n):
    if case == "sheared":  # the linearly mapped box of test_affine_geometry_kernel_on_a_sheared_box
        mesh = om.create_box(*n)
        M = np.array([[1.0, 0.3, -0.2], [0.1, 0.9, 0.25], [-0.15, 0.2, 1.1]])
        mesh.verts[:] = mesh.verts @ M.T + np.array([0.3, -1.0, 2.0])
        return mesh
    return om.create_box(*n, perturb=0.2 if case == "perturbed" else 0.0)


@pytest.mark.parametrize("P", [1, 2, 3, 4, 5, 6, 7, 8])
@pytest.mark.parametrize("case", ["perturbed", "uniform", "sheared"])
def test_recompute_apply_matches_oracle(ctx, P, case):
    n = (3, 4, 5) if P <= 4 else (2, 3, 2)
    mesh = _mesh(case, n)
    ol = OracleLevel(mesh, P)
    if case == "sheared":
        assert np.abs(ol.G[:, :, [1, 2, 4]]).max() > 1e-3
    rng = np.random.default_rng(42)
    # PMGX_LAP_STREAM_G has no effect together with the flag
    for flags in ((RECOMPUTE, RECOMPUTE | STREAM) if case == "uniform" else (RECOMPUTE,)):
        gl = GpuLevel(ctx, ol, flags=flags)
        assert gl.op.kernel_name() == KERNELS[P], gl.op.kernel_name()
        assert not gl.op.is_affine()
        for x in (rng.uniform(-1, 1, ol.nd), np.ones(ol.nd)):
            e2, einf = rel(gl.apply(x), ol.A(x))
            assert e2 < TOL and einf < TOL, (P, case, flags, e2, einf)
    if case == "perturbed":  # quirk Q17: the reference's literal det J expression
        oll = OracleLevel(mesh, P, literal_detj=True)
        gl = GpuLevel(ctx, oll, flags=RECOMPUTE | LITERAL)
        for x in (rng.uniform(-1, 1, ol.nd), np.ones(ol.nd)):
            e2, einf = rel(gl.apply(x), oll.A(x))
            assert e2 < TOL and einf < TOL, (P, "literal", e2, einf)


def _box_ops(ctx, P, n, perturb):
    """Default and recompute operators of one library-generated box (fast host set-up for large meshes)."""
    from pmg_dolfinx_b200 import api
    m = api.BoxMesh(n, perturb=perturb)
    s = m.space(P)
    d = dict(kappa=ctx.to_device(np.full(m.n_cells, 2.0)), dofmap=ctx.to_device(s.dofmap),
             xgeom=ctx.to_device(m.xgeom), gdm=ctx.to_device(m.geom_dofmap), bc=ctx.to_device(s.bc))
    ops = [api.MatFreeLaplacian(ctx, P, d["kappa"], d["dofmap"], d["xgeom"], d["gdm"], m.lcells, m.bcells, d["bc"],
                                s.n_owned, 0, None, flags) for flags in (0, RECOMPUTE)]
    return m, s, d, ops


def _apply(ctx, op, x):
    from pmg_dolfinx_b200 import api
    xv, yv = api.Vector(ctx, len(x)), api.Vector(ctx, len(x))
    xv.copy_from_host(x)
    op(xv, yv)
    return yv.data_copy()


# Sizes: every resident CTA (slab kernels) or warp (mma kernel) must process >= 3 batches / cells, so the rings,
# the double-buffered dofmap and the per-thread shared-memory columns wrap around several times.  The bounds
# assume more residency than the kernels have (148 SMs):
#   P1 slab: cpb = 64 / 2 = 32 cells per batch, <= 16 CTAs per SM: 3 * 32 * 16 * 148 = 227 328 cells -> 62^3
#   P4 slab: cpb = 128 / 5 = 25, <= 4 CTAs per SM (226 registers x 128 threads): 3 * 25 * 4 * 148 = 44 400 -> 36^3
#   P6 mma : one cell per warp, 2 warps per CTA, <= 8 CTAs per SM: 3 * 16 * 148 = 7 104 cells -> 20^3
#   P8 column (not persistent): cpb = 256 / 81 = 3 cells per CTA, <= 2 CTAs per SM: 21^3 cells = 3 087 CTAs are
#   >= 10 waves
@pytest.mark.parametrize("P,n", [(1, 62), (4, 36), (6, 20), (8, 21)])
def test_recompute_many_batches_per_cta(ctx, P, n):
    m, s, d, (op_d, op_r) = _box_ops(ctx, P, (n, n, n), 0.15)
    assert op_r.kernel_name() == KERNELS[P] and not op_d.is_affine()
    x = np.random.default_rng(P).uniform(-1, 1, s.n_owned)
    yd, yr = _apply(ctx, op_d, x), _apply(ctx, op_r, x)
    e2, einf = rel(yr, yd)
    assert e2 < TOL and einf < TOL, (P, e2, einf)
    if P == 1:  # and against the C oracle on the host
        from oracle import cport
        G, _ = cport.geometry(m.xgeom, m.geom_dofmap, P)
        yo = cport.Apply(P, s.dofmap, G, np.full(m.n_cells, 2.0), s.bc, s.n_owned)(x)
        e2, einf = rel(yr, yo)
        assert e2 < TOL and einf < TOL, (P, "oracle", e2, einf)


@pytest.mark.parametrize("P", [1, 3, 4, 6, 8])
def test_recompute_cell_lists_and_ragged_batches(ctx, P):
    ol = OracleLevel(om.create_box(3, 3, 5, perturb=0.15), P)
    rng = np.random.default_rng(7)
    perm = rng.permutation(ol.mesh.ncells).astype(np.int32)
    gl = GpuLevel(ctx, ol, flags=RECOMPUTE, lcells=perm[:17], bcells=perm[17:])
    x = rng.uniform(-1, 1, ol.nd)
    e2, einf = rel(gl.apply(x), ol.A(x))
    assert e2 < TOL and einf < TOL


def test_recompute_subset_of_cells_and_empty_lists(ctx):
    P = 2
    ol = OracleLevel(om.create_box(3, 3, 3, perturb=0.1), P)
    cells = np.array([0, 5, 13, 26], dtype=np.int32)
    gl = GpuLevel(ctx, ol, flags=RECOMPUTE, lcells=cells[:1], bcells=cells[1:])
    x = np.random.default_rng(3).uniform(-1, 1, ol.nd)
    yo = oo.apply_cells(P, ol.dm, ol.G, ol.kappa, ol.bc, x, np.zeros(ol.nd), cells)
    assert rel(gl.apply(x), yo)[0] < TOL
    g0 = GpuLevel(ctx, ol, flags=RECOMPUTE, lcells=np.zeros(0, np.int32), bcells=np.zeros(0, np.int32))
    assert np.abs(g0.apply(x)).max() == 0.0


@pytest.mark.parametrize("P", [1, 2, 3, 4, 5, 6, 7, 8])
def test_recompute_diagonal_matches_oracle(ctx, P):
    n = (3, 2, 3) if P <= 4 else (2, 2, 2)
    ol = OracleLevel(om.create_box(*n, perturb=0.2), P)
    gl = GpuLevel(ctx, ol, flags=RECOMPUTE)
    v = gl.vec()
    gl.op.get_diag_inverse(v)
    d = 1.0 / v.data_copy()
    do = ol.diag()
    assert np.abs(d - do).max() / np.abs(do).max() < 1e-13
    assert (d[ol.bc != 0] == 1.0).all()


@pytest.mark.parametrize("P", [1, 2, 4, 6, 8])
def test_recompute_geometry_factors_match_oracle(ctx, P):
    for literal in (False, True):
        ol = OracleLevel(om.create_box(2, 3, 2, perturb=0.2), P, literal_detj=literal)
        gl = GpuLevel(ctx, ol, flags=RECOMPUTE | (LITERAL if literal else 0))
        G = gl.op.geometry_factors()
        assert np.abs(G - ol.G).max() / np.abs(ol.G).max() < 1e-13


@pytest.mark.parametrize("P", [1, 2])
def test_recompute_csr_assembly(ctx, P):
    ol = OracleLevel(om.create_box(4, 3, 5, perturb=0.2), P)
    Ao = oo.assemble_csr(P, ol.dm, ol.G, ol.kappa, ol.bc, ol.nd)
    mats = []
    for flags in (0, RECOMPUTE):
        rp, co, va = GpuLevel(ctx, ol, flags=flags).op.to_csr().to_host()
        mats.append((rp, co, va))
    (rp0, co0, va0), (rp1, co1, va1) = mats
    assert np.array_equal(rp0, rp1) and np.array_equal(co0, co1)
    Ag = sp.csr_matrix((va1, co1, rp1), shape=(ol.nd, ol.nd))
    assert abs(Ag - Ao).max() < 1e-13 * abs(Ao).max()
    assert np.abs(va1 - va0).max() < 1e-13 * np.abs(va0).max()


@pytest.mark.parametrize("P", [1, 3, 6])
def test_recompute_rhs_with_lifting(ctx, P):
    mesh = om.create_box(4, 3, 5, perturb=0.15)
    ol = OracleLevel(mesh, P, kappa=np.random.default_rng(3).uniform(0.5, 2.0, mesh.ncells))
    gl = GpuLevel(ctx, ol, flags=RECOMPUTE)
    X = om.dof_coords(mesh, P)
    f = lambda Y: 1000.0 * np.exp(-((Y[:, 0] - 0.5) ** 2 + (Y[:, 1] - 0.5) ** 2) / 0.02)
    bo = oo.rhs_collocated(mesh, P, f, ol.bc, g=1.3, kappa=ol.kappa)
    bv = gl.vec()
    gl.op.assemble_rhs(ctx.to_device(f(X)), 1.3, bv)
    assert rel(bv.data_copy(), bo)[0] < TOL
    gvec = np.where(ol.bc != 0, 1.0 + X[:, 0] - 2.0 * X[:, 2], 7.0)
    bo2 = oo.rhs_collocated(mesh, P, f, ol.bc, g=gvec, kappa=ol.kappa)
    bv2 = gl.vec()
    gl.op.assemble_rhs(ctx.to_device(f(X)), 0.0, bv2)
    gl.op.lift(ctx.to_device(gvec), bv2)
    assert rel(bv2.data_copy(), bo2)[0] < TOL


def test_recompute_device_memory(ctx):
    """P1, 10^6 cells: the default operator holds >= 384 B of G per cell; the recompute operator only the encoded
    dofmap (32 B per cell with its batch padding), perm and the inverse diagonal.  Both agree with the free-memory
    drop around create."""
    from pmg_dolfinx_b200 import api
    P, n = 1, 100
    m = api.BoxMesh((n, n, n), perturb=0.15)
    s = m.space(P)
    kappa, dofmap = ctx.to_device(np.full(m.n_cells, 2.0)), ctx.to_device(s.dofmap)
    xgeom, gdm, bc = ctx.to_device(m.xgeom), ctx.to_device(m.geom_dofmap), ctx.to_device(s.bc)
    nc = m.n_cells
    assert nc >= 10 ** 6
    got = {}
    for flags in (0, RECOMPUTE):
        ctx.sync()
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        op = api.MatFreeLaplacian(ctx, P, kappa, dofmap, xgeom, gdm, m.lcells, m.bcells, bc, s.n_owned, 0, None, flags)
        ctx.sync()
        free1 = torch.cuda.mem_get_info()[0]
        got[flags] = (op.device_bytes(), free0 - free1)
        op.destroy()
    (bd, dd), (br, dr) = got[0], got[RECOMPUTE]
    assert bd >= 384 * nc
    nbatch = -(-len(m.lcells) // 32) + -(-len(m.bcells) // 32)
    bound = nbatch * 4 * 64 * 4 + 4 * nc + 8 * s.n_owned + 4096
    assert br <= bound, (br, bound)
    assert bd - br >= 384 * nc
    for b, delta in ((bd, dd), (br, dr)):  # cudaMalloc granularity: 2 MiB per allocation, a handful of them
        assert abs(delta - b) <= 16 * 2 ** 20, (b, delta)


def test_recompute_sees_vertices_moved_in_place(ctx):
    P = 3
    mesh = om.create_box(3, 4, 5, perturb=0.1)
    ol = OracleLevel(mesh, P)
    gl = GpuLevel(ctx, ol, flags=RECOMPUTE)
    x = np.random.default_rng(11).uniform(-1, 1, ol.nd)
    assert rel(gl.apply(x), ol.A(x))[1] < TOL
    V = mesh.verts
    interior = np.all((V > V.min(axis=0) + 1e-9) & (V < V.max(axis=0) - 1e-9), axis=1)
    assert interior.sum() > 10
    disp = np.zeros_like(V)
    disp[interior] = np.random.default_rng(12).uniform(-0.04, 0.04, (interior.sum(), 3))
    gl.xgeom += ctx.to_device(disp)  # in place, on the device
    mesh2 = om.create_box(3, 4, 5, perturb=0.1)
    mesh2.verts[:] = V + disp
    ol2 = OracleLevel(mesh2, P)
    y = gl.apply(x)
    assert rel(y, ol.A(x))[1] > 1e-6
    e2, einf = rel(y, ol2.A(x))
    assert e2 < TOL and einf < TOL


def _vcycle_residuals(ctx, ols, flags, lmax):
    from pmg_dolfinx_b200 import api
    gls = [GpuLevel(ctx, ol, flags=flags) for ol in ols]
    smoothers = []
    for ol, lm in zip(ols, lmax):
        s = api.Chebyshev(ctx, ol.nd, 0, (0.1 * lm / 1.1, lm))
        s.set_max_iterations(2)
        smoothers.append(s)
    allc = np.arange(ols[0].mesh.ncells, dtype=np.int32)
    interps = [api.Interpolator(ctx, a.P, b.P, ga.dofmap, gb.dofmap, a.nd, b.nd, allc, allc[:0])
               for a, b, ga, gb in zip(ols[:-1], ols[1:], gls[:-1], gls[1:])]
    pmg = api.MultigridPreconditioner(ctx, [g.bc for g in gls], flags=2)
    pmg.set_solvers(smoothers)
    pmg.set_operators([g.op for g in gls])
    pmg.set_interpolators(interps)
    pmg.set_coarse_solver(None)
    top = ols[-1]
    b = oo.rhs_collocated(top.mesh, top.P, oo.f_sines(1, 1, 1, 2.0), top.bc)
    u, bv = gls[-1].vec(), gls[-1].vec(b)
    out = []
    for _ in range(3):
        out.append(pmg.apply(bv, u, verbose=True))
        out.extend(pmg.diagnostics())
    return np.array(out)


def test_recompute_vcycle_hierarchy_matches_default(ctx):
    mesh = om.create_box(4, 4, 4, perturb=0.15)
    ols = [OracleLevel(mesh, P) for P in (1, 2, 4)]
    lmax = []
    for ol in ols:
        _, _, al, be, _, _ = osol.cg(ol.A, 1.0 / ol.diag(), np.zeros(ol.nd), np.ones(ol.nd), 20, 1e-6)
        lmax.append(1.1 * osol.lanczos_eigenvalues(al, be)[-1])
    hd = _vcycle_residuals(ctx, ols, 0, lmax)
    hr = _vcycle_residuals(ctx, ols, RECOMPUTE, lmax)
    assert len(hd) == len(hr) and np.all(np.abs(hr - hd) <= 1e-10 * np.abs(hd)), (hd, hr)


def test_recompute_jacobi_cg_matches_default(ctx):
    from pmg_dolfinx_b200 import api
    ol = OracleLevel(om.create_box(4, 5, 3, perturb=0.2), 3)
    hist = []
    for flags in (0, RECOMPUTE):
        gl = GpuLevel(ctx, ol, flags=flags)
        cg = api.CGSolver(ctx, ol.nd, 0)
        cg.set_max_iterations(200)
        cg.set_tolerance(1e-8)
        x = gl.vec()
        k = cg.solve(gl.op, x, gl.vec(np.ones(ol.nd)))
        hist.append((k, cg.history()))
    (kd, (r0d, hd)), (kr, (r0r, hr)) = hist
    assert kd == kr and kd < 200
    assert abs(r0r - r0d) <= 1e-10 * r0d
    assert len(hd) == len(hr) and np.all(np.abs(hr - hd) <= 1e-10 * np.abs(hd))


def test_cpp_pmg_driver_with_batch_size(ctx):
    """The shim accepts batch_size > 0: ten V-cycle residuals equal the default run's to 1e-8 relative."""
    r = subprocess.run(["make"], cwd=os.path.join(ROOT, "examples"), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    pmg = os.path.join(ROOT, "examples", "build", "pmg_main")
    res = []
    for extra in ([], ["--batch_size", "1"]):
        r = subprocess.run([pmg, "--ndofs", "40000", "--perturb", "0.15", "--niter", "10"] + extra,
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        res.append(np.array([float(v) for v in re.findall(r"relative ([0-9.eE+-]+)\)", r.stdout)]))
    assert len(res[0]) == 10 and len(res[1]) == 10
    assert np.all(np.abs(res[1] - res[0]) <= 1e-8 * res[0]), res
