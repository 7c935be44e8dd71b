"""GPU parity of two CSR paths that the other tests never reach: the ghost-column block on one GPU, and the 32-bit
columns of the sliced-ELL smoother matrix.

Ghost columns: a MatrixOperator whose rows have entries after off_diag_offset runs k_spmv_ghost_rows in the SpMV
and, in the fused Chebyshev solve, parks the owned-column partial sum of those rows in a scratch vector and finishes
them in k_spmv_cheb_ghost_rows.  The Chebyshev test takes two such matrices: one built from host arrays, and the P1
matrix of one rank of a box partition, assembled on the device with its ghost-column block (pmgx_csr_from_laplacian).
Without a halo the ghost block of x is whatever the caller put there, and the smoother's internal vectors keep a zero
ghost block (they are zeroed at allocation), so the solve is the Chebyshev iteration of A_oo with right-hand side
b - A_og x_g.

32-bit columns: the AMG level-0 smoother matrix stores FP32 values with 16-bit column deltas, and falls back to 32-bit
columns when some owned-column delta leaves +-32767.  A randomly permuted P1 matrix has such deltas.

Not covered: the parked-sum branch inside k_spmv_sell_cheb (off_diag non-null).  The AMG host set-up takes no ghost
columns on a single rank, so it needs a preconditioner-application test on several GPUs.
"""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla
import torch

from oracle import mesh as om, operator as oo, solvers as osol

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))


def _ghost_problem(seed=4):
    """The oracle's P1 matrix on a perturbed box with a scattered subset of its dofs declared ghosts: (the owned rows
    [A_oo A_og] as CSR with owned columns first in each row, owned count, ghost count, off_diag_offset)"""
    m = om.create_box(6, 5, 7, perturb=0.15)
    G, _ = oo.geometry_factors(m.verts, m.geom_dofmap, 1)
    dm, bc, nd = om.dofmap(m, 1), om.bc_marker(m, 1), om.num_dofs(m, 1)
    kap = np.random.default_rng(seed).uniform(0.5, 2.0, m.ncells)
    A = oo.assemble_csr(1, dm, G, kap, bc, nd)
    rng = np.random.default_rng(seed)
    ghost = np.zeros(nd, dtype=bool)
    ghost[rng.choice(nd, nd // 5, replace=False)] = True
    order = np.concatenate([rng.permutation(np.flatnonzero(~ghost)), rng.permutation(np.flatnonzero(ghost))])
    n_o = int((~ghost).sum())
    R = sp.csr_matrix(A[order][:, order][:n_o])   # rows: owned dofs; columns: owned, then ghosts
    R.sort_indices()                              # sorted columns: the owned block comes first in each row
    rows = np.repeat(np.arange(n_o), np.diff(R.indptr))
    off = R.indptr[:-1] + np.bincount(rows[R.indices < n_o], minlength=n_o)
    return R, n_o, nd - n_o, off.astype(np.int32)


def test_ghost_problem_has_rows_with_and_without_ghost_columns():
    R, n_o, k, off = _ghost_problem()
    has = off < R.indptr[1:]
    assert 0.2 * n_o < has.sum() < 0.9 * n_o
    for i in np.flatnonzero(has)[:50]:
        c = R.indices[R.indptr[i]:R.indptr[i + 1]]
        assert (c[: off[i] - R.indptr[i]] < n_o).all() and (c[off[i] - R.indptr[i]:] >= n_o).all()


def _ghost_operator(ctx):
    from pmg_dolfinx_b200 import api
    R, n_o, k, off = _ghost_problem()
    op = api.MatrixOperator(ctx, R.indptr, off, R.indices, R.data, n_ghost=k, halo=None)
    return api, R, n_o, k, op


def _device_ghost_operator(ctx):
    """rank 0 of a (2, 1, 1) partition of a perturbed box: its P1 matrix assembled on the device, as (api, the owned
    rows [A_oo A_og], owned count, ghost count, operator)"""
    from pmg_dolfinx_b200 import api
    m = api.BoxMesh((6, 5, 7), (2, 1, 1), 0, perturb=0.15)
    s = m.space(1)
    kap = np.random.default_rng(4).uniform(0.5, 2.0, m.n_cells)
    d = [ctx.to_device(a) for a in (kap, s.dofmap, m.xgeom, m.geom_dofmap, s.bc)]
    lap = api.MatFreeLaplacian(ctx, 1, d[0], d[1], d[2], d[3], m.lcells, m.bcells, d[4], s.n_owned, s.n_ghost)
    op = lap.to_csr()
    m.close()
    rp, co, va = op.to_host()
    R = sp.csr_matrix((va, co, rp), shape=(s.n_owned, s.n_owned + s.n_ghost))
    assert s.n_ghost > 0 and R[:, s.n_owned:].nnz > 0
    return api, R, s.n_owned, s.n_ghost, op


def _vec(api, ctx, n_o, k, owned, ghost):
    v = api.Vector(ctx, n_o, k)
    v.data[:n_o].copy_(torch.from_numpy(np.ascontiguousarray(owned)))
    v.data[n_o:].copy_(torch.from_numpy(np.ascontiguousarray(ghost)))
    return v


def test_spmv_with_ghost_columns_and_no_halo(ctx):
    api, R, n_o, k, op = _ghost_operator(ctx)
    assert op.n_owned == n_o and op.n_ghost == k
    rng = np.random.default_rng(1)
    xo, xg = rng.uniform(-1, 1, n_o), rng.uniform(-1, 1, k)
    yv = _vec(api, ctx, n_o, k, np.full(n_o, np.nan), np.full(k, 5.0))
    op(_vec(api, ctx, n_o, k, xo, xg), yv)
    y = yv.data_copy()
    yo = R @ np.concatenate([xo, xg])
    assert np.abs(y[:n_o] - yo).max() <= 1e-14 * np.abs(yo).max()
    assert (y[n_o:] == 0.0).all()                 # ghost entries of y are zeroed
    # the ghost block really contributes
    assert np.abs(R[:, n_o:] @ xg).max() > 0.1 * np.abs(yo).max()


@pytest.mark.parametrize("its", [2, 3, 5])
@pytest.mark.parametrize("x0", ["zero", "nonzero"])
@pytest.mark.parametrize("matrix", ["host", "device"])
def test_chebyshev_with_ghost_columns_fused_and_unfused(ctx, its, x0, matrix):
    """silent solve: the fused path (k_spmv_cheb + k_spmv_cheb_ghost_rows with the parked sums); verbose solve: the
    unfused path (SpMV, then a vector pass).  Both against the oracle's Chebyshev on A_oo, b - A_og x_g."""
    api, R, n_o, k, op = (_ghost_operator if matrix == "host" else _device_ghost_operator)(ctx)
    Aoo, Aog = R[:, :n_o].tocsr(), R[:, n_o:].tocsr()
    dinv = 1.0 / Aoo.diagonal()
    dv = api.Vector(ctx, n_o, k)
    op.get_diag_inverse(dv)
    assert np.allclose(dv.data_copy()[:n_o], dinv, rtol=1e-15, atol=0)
    _, _, al, be, _, _ = osol.cg(lambda v: Aoo @ v, dinv, np.zeros(n_o), np.ones(n_o), 20, 1e-6)
    lmax = 1.1 * osol.lanczos_eigenvalues(al, be)[-1]
    rng = np.random.default_rng(10 * its + (x0 == "zero"))
    b, xg = rng.uniform(-1, 1, n_o), rng.uniform(-1, 1, k)
    x0o = np.zeros(n_o) if x0 == "zero" else rng.uniform(-1, 1, n_o)
    ho = []
    xo = osol.chebyshev(lambda v: Aoo @ v, dinv, x0o, b - Aog @ xg, its, lmax, history=ho)
    ch = api.Chebyshev(ctx, n_o, k, (0.1 * lmax / 1.1, lmax))
    ch.set_max_iterations(its)
    out = {}
    for verbose in (False, True, False):           # fused, unfused, fused again after the unfused solve
        xv = _vec(api, ctx, n_o, k, x0o, xg)
        bv = _vec(api, ctx, n_o, k, b, np.zeros(k))
        h = ch.solve(op, xv, bv, verbose=verbose)
        x = xv.data_copy()
        assert np.array_equal(x[n_o:], xg)         # the ghost block of x is read, never written
        if verbose:
            assert np.all(np.abs(h - np.array(ho)) <= 1e-12 * np.array(ho)), (h, ho)
        err = np.linalg.norm(x[:n_o] - xo) / np.linalg.norm(xo)
        assert err < 1e-13, (its, x0, verbose, err)
        out.setdefault(verbose, []).append(x[:n_o])
    fused, unfused = out[False][0], out[True][0]
    assert np.abs(fused - unfused).max() <= 1e-14 * np.abs(unfused).max()
    assert np.array_equal(out[False][0], out[False][1])


# ---- 32-bit columns of the sliced-ELL level-0 smoother matrix
N32 = 32   # p1_matrix(32): 33^3 = 35 937 rows


@pytest.fixture(scope="module")
def permuted_p1():
    import prototype_sa_amg as proto
    A, bc = proto.p1_matrix(N32)
    p = np.random.default_rng(8).permutation(A.shape[0])
    Ap = sp.csr_matrix(A[p][:, p])
    Ap.sort_indices()
    return Ap, bc[p]


def test_permuted_matrix_needs_32_bit_columns(permuted_p1):
    """the condition under which the level-0 smoother matrix keeps 32-bit columns, on the pattern it streams (stored
    zeros dropped, diagonal kept)"""
    import prototype_sa_amg as proto
    from test_gpu_coarse_sparsity import _nonzeros
    A, _ = permuted_p1
    assert A.shape[0] == 35937
    Z = _nonzeros(A)
    rows = np.repeat(np.arange(Z.shape[0]), np.diff(Z.indptr))
    assert np.abs(Z.indices.astype(np.int64) - rows).max() > 32767
    nat, _ = proto.p1_matrix(N32)
    Zn = _nonzeros(sp.csr_matrix(nat))
    rn = np.repeat(np.arange(Zn.shape[0]), np.diff(Zn.indptr))
    assert np.abs(Zn.indices.astype(np.int64) - rn).max() <= 32767   # natural order: 16-bit deltas suffice


def _coarse(ctx, A, nu=2):
    from pmg_dolfinx_b200 import api
    op = api.MatrixOperator(ctx, A.indptr, A.indptr[1:], A.indices, A.data)
    return api, op, api.CoarseSolverType(ctx, op, 60, 1e-8, amg=True, nu=nu, min_coarse=100)


@pytest.mark.parametrize("nu", [1, 2, 3, 4])
def test_preconditioner_on_a_matrix_with_32_bit_columns(ctx, permuted_p1, nu):
    """nu = 1: the stand-alone SpMV k_spmv_sell<false>; nu >= 2: the fused k_spmv_sell_cheb<false, *>"""
    import prototype_sa_amg as proto
    from test_amg_setup import _hierarchy, _fp32_level0
    A, bc = permuted_p1
    nd = A.shape[0]
    api, op, cs = _coarse(ctx, A, nu)
    levels = _hierarchy(A, min_coarse=100, max_levels=12)
    info = cs.levels()
    assert len(info) == len(levels) and [i[0] for i in info] == [l["A"].shape[0] for l in levels]
    rng = np.random.default_rng(3)
    r = rng.uniform(-1, 1, nd) * (~bc)
    rv, uv = api.Vector(ctx, nd), api.Vector(ctx, nd)
    rv.copy_from_host(r)
    cs.apply_preconditioner(rv, uv)
    u = uv.data_copy()
    uo = proto.vcycle(_fp32_level0(levels), 0, r, nu)
    assert np.linalg.norm(u - uo) <= 1e-10 * np.linalg.norm(uo), np.linalg.norm(u - uo) / np.linalg.norm(uo)
    s = rng.uniform(-1, 1, nd) * (~bc)
    sv, tv = api.Vector(ctx, nd), api.Vector(ctx, nd)
    sv.copy_from_host(s)
    cs.apply_preconditioner(sv, tv)
    a, b = float(np.dot(s, u)), float(np.dot(r, tv.data_copy()))
    assert abs(a - b) <= 1e-10 * max(abs(a), abs(b))


def test_pcg_on_a_matrix_with_32_bit_columns(ctx, permuted_p1):
    A, bc = permuted_p1
    nd = A.shape[0]
    api, op, cs = _coarse(ctx, A)
    b = np.random.default_rng(1).uniform(-1, 1, nd) * (~bc)
    bv, xv = api.Vector(ctx, nd), api.Vector(ctx, nd)
    bv.copy_from_host(b)
    k = cs.solve(xv, bv)
    conv, relres = cs.last_status()
    assert conv and relres < 1e-8 and k <= 12, (k, conv, relres)
    xo = spla.spsolve(sp.csc_matrix(A), b)
    assert np.linalg.norm(xv.data_copy() - xo) <= 1e-7 * np.linalg.norm(xo)
