"""GPU: the device cycle of the smoothed-aggregation coarse solver (csrc/amg.cu) behind
CoarseSolverType::solve (src/amg.hpp:67-113: PETSc KSPCG + BoomerAMG in the reference).

The reference holds no numbers for this third-party solve, so the device cycle is pinned against the
numpy V-cycle of scripts/prototype_sa_amg.py run on the SAME hierarchy (pulled back from the library's
host set-up, which tests/test_amg_setup.py and tests/test_amg_dist_cpu.py check against scipy), with level 0's
smoothing matrix rounded to FP32 as the device streams it: one application u = M^-1 r to 1e-10, symmetry of
M^-1, and the PCG solve against scipy's direct solution."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _setup(ctx, n, min_coarse, nu=2, rtol=1e-8, max_iter=60):
    from pmg_dolfinx_b200 import api
    import prototype_sa_amg as proto
    A, bc = proto.p1_matrix(n)
    A = sp.csr_matrix(A)
    A.sort_indices()
    nd = A.shape[0]
    op = api.MatrixOperator(ctx, A.indptr, A.indptr[1:], A.indices, A.data)   # no ghost columns: off_diag = row end
    cs = api.CoarseSolverType(ctx, op, max_iter, rtol, amg=True, nu=nu, min_coarse=min_coarse)
    return api, proto, A, bc, nd, op, cs


@pytest.mark.parametrize("nu", [1, 2, 3, 4])
@pytest.mark.parametrize("n", [6, 8, 12, 16, 20, 24])
def test_device_cycle_equals_numpy_cycle_on_the_same_hierarchy(ctx, n, nu):
    """The level-0 smoother streams the matrix with FP32 values and 16-bit column deltas, so the device cycle is the
    exact cycle of the hierarchy with level 0's smoothing matrix rounded to FP32.  nu = 1 runs the stand-alone SpMVs
    and vector passes of the smoother (csr.cu k_spmv_sell, k_spmv); nu >= 2 runs the SpMVs with the Chebyshev update
    as their epilogue on every level (k_spmv_sell_cheb, k_spmv_cheb), nu >= 3 with more than one z swap."""
    from test_amg_setup import _hierarchy, _fp32_level0
    api, proto, A, bc, nd, op, cs = _setup(ctx, n, 100, nu=nu)
    levels = _hierarchy(A, min_coarse=100, max_levels=12)
    info = cs.levels()
    assert len(info) == len(levels) and info[-1][3] == 1
    assert [i[4] for i in info[:-1]] == [l["P"].nnz for l in levels[:-1]]
    assert [i[0] for i in info] == [l["A"].shape[0] for l in levels]
    assert [i[1] for i in info] == [l["A"].nnz for l in levels]
    rng = np.random.default_rng(3)
    r = rng.uniform(-1, 1, nd) * (~bc)
    rv, uv = api.Vector(ctx, nd), api.Vector(ctx, nd)
    rv.copy_from_host(r)
    cs.apply_preconditioner(rv, uv)
    u = uv.data_copy()
    uo = proto.vcycle(_fp32_level0(levels), 0, r, nu)
    assert np.linalg.norm(u - uo) <= 1e-10 * np.linalg.norm(uo), np.linalg.norm(u - uo) / np.linalg.norm(uo)
    # M^-1 is symmetric (same Chebyshev polynomial before and after the coarse correction)
    s = rng.uniform(-1, 1, nd) * (~bc)
    sv, tv = api.Vector(ctx, nd), api.Vector(ctx, nd)
    sv.copy_from_host(s)
    cs.apply_preconditioner(sv, tv)
    a, b = float(np.dot(s, u)), float(np.dot(r, tv.data_copy()))
    assert abs(a - b) <= 1e-10 * max(abs(a), abs(b))   # the rounded matrix is symmetric too


@pytest.mark.parametrize("n", [12, 24])
def test_amg_pcg_converges_in_a_handful_of_iterations(ctx, n):
    api, proto, A, bc, nd, op, cs = _setup(ctx, n, 100, rtol=1e-8)
    b = np.random.default_rng(1).uniform(-1, 1, nd) * (~bc)
    bv, xv = api.Vector(ctx, nd), api.Vector(ctx, nd)
    bv.copy_from_host(b)
    k = cs.solve(xv, bv)
    conv, relres = cs.last_status()
    assert conv and relres < 1e-8 and k <= 12, (k, conv, relres)
    xo = spla.spsolve(sp.csc_matrix(A), b)
    x = xv.data_copy()
    assert np.linalg.norm(x - xo) <= 1e-7 * np.linalg.norm(xo)
    # Jacobi-PCG on the same operator needs an order of magnitude more iterations -- and says so when capped
    cj = api.CoarseSolverType(ctx, op, 16, 1e-8, amg=False)
    xj = api.Vector(ctx, nd)
    kj = cj.solve(xj, bv)
    assert kj == 16 and not cj.last_status()[0] and cj.last_status()[1] > 1e-8


def test_single_level_hierarchy_is_a_direct_solve(ctx):
    api, proto, A, bc, nd, op, cs = _setup(ctx, 6, 600, rtol=1e-12)
    assert len(cs.levels()) == 1 and cs.levels()[0][3] == 1
    b = np.random.default_rng(5).uniform(-1, 1, nd)
    bv, xv = api.Vector(ctx, nd), api.Vector(ctx, nd)
    bv.copy_from_host(b)
    k = cs.solve(xv, bv)
    assert k <= 2 and cs.last_status()[0]
    assert np.linalg.norm(xv.data_copy() - spla.spsolve(sp.csc_matrix(A), b)) <= 1e-11 * np.linalg.norm(b)
