"""GPU: the AMG coarse solver on an assembled P1 matrix that carries stored zeros.

pmgx_csr_from_laplacian keeps the full 27-entry element pattern; with the collocated GLL quadrature an interior
row of a uniform box has 7 non-zeros (about 16 on a perturbed box).  The hierarchy is built from that full
pattern, while PCG, the level-0 smoother and the level-0 transfers stream copies without the zeros.  These
tests pin the solver on such a matrix against the numpy cycle of scripts/prototype_sa_amg.py on the hierarchy
of the full pattern, and the PCG solve against scipy."""
import ctypes
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

BOXES = [0.0, 0.15]
BOX_IDS = ["uniform-box", "perturbed-box"]


def _p1_csr(ctx, perturb, n=16):
    """the device-assembled P1 operator (stored zeros included) and the same matrix on the host"""
    from pmg_dolfinx_b200 import api
    from oracle import mesh as om
    m = om.create_box(n, n, n, perturb=perturb)
    dm, bc, nd = om.dofmap(m, 1), om.bc_marker(m, 1), om.num_dofs(m, 1)
    d_dm, d_x, d_g = ctx.to_device(dm), ctx.to_device(m.verts), ctx.to_device(m.geom_dofmap)
    d_k, d_bc = ctx.to_device(np.full(m.ncells, 2.0)), ctx.to_device(bc)
    cells = np.arange(m.ncells, dtype=np.int32)
    op = api.MatFreeLaplacian(ctx, 1, d_k, d_dm, d_x, d_g, cells, cells[:0], d_bc, nd)
    A = op.to_csr()
    rp, co, va = A.to_host()
    H = sp.csr_matrix((va, co, rp), shape=(nd, nd))   # keeps the explicit zeros
    H.sort_indices()
    return api, A, H, np.asarray(bc, dtype=bool), nd


def _nonzeros(H):
    """H without its stored zeros, filtered by the library's host filter"""
    from pmg_dolfinx_b200.capi import lib, check, ptr
    n = H.shape[0]
    ip, ix = H.indptr.astype(np.int32), H.indices.astype(np.int32)
    kept = ctypes.c_longlong(0)
    check(lib.pmgx_csr_drop_zeros_h(n, ptr(ip), ptr(ix), ptr(H.data), None, None, None, ctypes.addressof(kept)))
    op, oc, ov = np.zeros(n + 1, np.int32), np.zeros(kept.value, np.int32), np.zeros(kept.value)
    check(lib.pmgx_csr_drop_zeros_h(n, ptr(ip), ptr(ix), ptr(H.data), ptr(op), ptr(oc), ptr(ov), ctypes.addressof(kept)))
    return sp.csr_matrix((ov, oc, op), shape=H.shape)


@pytest.mark.parametrize("perturb", BOXES, ids=BOX_IDS)
def test_hierarchy_is_built_from_the_full_pattern(ctx, perturb):
    from test_amg_setup import _hierarchy
    api, A, H, bc, nd = _p1_csr(ctx, perturb)
    Z = _nonzeros(H)
    assert Z.nnz * 5 <= H.nnz * 4                         # enough zeros for the solver to stream the copy
    assert abs(Z - H).max() == 0.0
    cs = api.CoarseSolverType(ctx, A, 60, 1e-8, amg=True, nu=2, min_coarse=100)
    levels = _hierarchy(H, min_coarse=100, max_levels=12)
    info = cs.levels()
    assert info[0][1] == H.nnz                            # level 0 reports the assembled pattern
    assert [i[0] for i in info] == [l["A"].shape[0] for l in levels]
    assert [i[1] for i in info] == [l["A"].nnz for l in levels]
    assert [i[4] for i in info[:-1]] == [l["P"].nnz for l in levels[:-1]]


@pytest.mark.parametrize("fuse_from", [0, 1, 99], ids=["fused-smoother-all-levels", "fused-from-level-1", "unfused"])
@pytest.mark.parametrize("lp", [False, True], ids=["fp64-matrix", "fp32-int16-smoother-matrix"])
@pytest.mark.parametrize("perturb", BOXES, ids=BOX_IDS)
def test_preconditioner_equals_numpy_cycle_of_the_full_pattern(ctx, perturb, lp, fuse_from, monkeypatch):
    import prototype_sa_amg as proto
    from test_amg_setup import _hierarchy
    monkeypatch.setenv("PMGX_AMG_LP", "1" if lp else "0")
    monkeypatch.setenv("PMGX_AMG_FUSE_FROM", str(fuse_from))
    api, A, H, bc, nd = _p1_csr(ctx, perturb)
    cs = api.CoarseSolverType(ctx, A, 60, 1e-8, amg=True, nu=2, min_coarse=100)
    levels = _hierarchy(H, min_coarse=100, max_levels=12)
    rng = np.random.default_rng(7)
    r = rng.uniform(-1, 1, nd) * (~bc)
    rv, uv = api.Vector(ctx, nd), api.Vector(ctx, nd)
    rv.copy_from_host(r)
    cs.apply_preconditioner(rv, uv)
    u = uv.data_copy()
    uo = proto.vcycle(levels, 0, r, 2)
    tol = 2e-6 if lp else 1e-10
    assert np.linalg.norm(u - uo) <= tol * np.linalg.norm(uo)
    s = rng.uniform(-1, 1, nd) * (~bc)
    sv, tv = api.Vector(ctx, nd), api.Vector(ctx, nd)
    sv.copy_from_host(s)
    cs.apply_preconditioner(sv, tv)
    a, b = float(np.dot(s, u)), float(np.dot(r, tv.data_copy()))
    assert abs(a - b) <= 1e-10 * max(abs(a), abs(b))


@pytest.mark.parametrize("perturb", BOXES, ids=BOX_IDS)
def test_pcg_matches_the_full_pattern_solve(ctx, perturb):
    import prototype_sa_amg as proto
    from test_amg_setup import _hierarchy
    api, A, H, bc, nd = _p1_csr(ctx, perturb)
    cs = api.CoarseSolverType(ctx, A, 60, 1e-8, amg=True, nu=2, min_coarse=100)
    b = np.random.default_rng(1).uniform(-1, 1, nd) * (~bc)
    bv, xv = api.Vector(ctx, nd), api.Vector(ctx, nd)
    bv.copy_from_host(b)
    k = cs.solve(xv, bv)
    conv, relres = cs.last_status()
    assert conv and relres < 1e-8
    # PCG on the full-pattern matrix with the numpy cycle of the same hierarchy takes as many iterations
    levels = _hierarchy(H, min_coarse=100, max_levels=12)
    _, k_full = proto.pcg(H, b, lambda r: proto.vcycle(levels, 0, r, 2), 1e-8, 60)
    assert k == k_full, (k, k_full)
    xo = spla.spsolve(sp.csc_matrix(H), b)
    assert np.linalg.norm(xv.data_copy() - xo) <= 1e-7 * np.linalg.norm(xo)
