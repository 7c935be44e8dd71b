"""Host set-up of the smoothed-aggregation hierarchy (pmgx_amg_setup_h, csrc/amg_setup.cpp; CPU only).
The level matrices built by the C++ code are pulled back and checked against scipy (Galerkin
identity, prolongator structure) and used in the numpy V-cycle of scripts/prototype_sa_amg.py: the
PCG iteration counts must be the mesh-independent handful the prototype shows, far below Jacobi-PCG."""
import ctypes
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
import prototype_sa_amg as proto  # noqa: E402
from pmg_dolfinx_b200.capi import lib, check, ptr  # noqa: E402


def _hierarchy(A, min_coarse=400, max_levels=10):
    A = sp.csr_matrix(A)
    A.sort_indices()
    h = ctypes.c_void_p()
    ip, ix = A.indptr.astype(np.int32), A.indices.astype(np.int32)
    check(lib.pmgx_amg_setup_h(A.shape[0], ptr(ip), ptr(ix), ptr(A.data), min_coarse, max_levels, ctypes.addressof(h)))
    levels = []
    for l in range(lib.pmgx_amg_num_levels(h)):
        sz = np.zeros(4, dtype=np.int64)
        check(lib.pmgx_amg_level_sizes(h, l, ptr(sz)))
        n, nnz, pc, pnnz = (int(v) for v in sz)
        ap, ac, av = np.zeros(n + 1, np.int32), np.zeros(nnz, np.int32), np.zeros(nnz)
        pp, pcl, pv = np.zeros(n + 1, np.int32), np.zeros(pnnz, np.int32), np.zeros(pnnz)
        lmax = ctypes.c_double()
        check(lib.pmgx_amg_level_get(h, l, ptr(ap), ptr(ac), ptr(av), ptr(pp) if pc else None,
                                     ptr(pcl) if pc else None, ptr(pv) if pc else None, ctypes.addressof(lmax)))
        lev = dict(A=sp.csr_matrix((av, ac, ap), shape=(n, n)), lmax=lmax.value)
        lev["dinv"] = 1.0 / lev["A"].diagonal()
        if pc:
            lev["P"] = sp.csr_matrix((pv, pcl, pp), shape=(n, pc))
        levels.append(lev)
    check(lib.pmgx_amg_destroy(h))
    levels[-1]["dense"] = np.linalg.inv(levels[-1]["A"].toarray())
    return levels


def _fp32_level0(levels):
    """The hierarchy as the device cycle runs it: level 0 smooths with its matrix rounded to FP32 (the sliced-ELL copy
    of csrc/csr.cu, make_lp), and the restriction takes the smoother's residual.  Its dinv and lmax, the transfers and
    the coarser levels stay FP64."""
    A = levels[0]["A"].copy()
    A.data = A.data.astype(np.float32).astype(np.float64)
    return [dict(levels[0], A=A)] + levels[1:]


@pytest.mark.parametrize("n", [8, 16, 24])
def test_hierarchy_is_galerkin_and_converges_like_the_prototype(n):
    A, bc = proto.p1_matrix(n)
    levels = _hierarchy(A, min_coarse=100)
    assert len(levels) >= 2 and levels[-1]["A"].shape[0] <= 100
    for fine, coarse in zip(levels[:-1], levels[1:]):
        P = fine["P"]
        G = (P.T @ fine["A"] @ P).tocsr()
        assert abs(G - coarse["A"]).max() <= 1e-12 * abs(G).max()           # A_c = P^T A P
        assert abs(coarse["A"] - coarse["A"].T).max() <= 1e-12 * abs(G).max()  # symmetric
        # Dirichlet rows (only a diagonal entry) carry no prolongator entries; every free row does
        free = np.diff(fine["A"].indptr) > 1
        rows_with_p = np.diff(P.indptr) > 0
        assert (rows_with_p[free]).all() and not rows_with_p[~free].any()
        # lambda_max estimate bounds the power-iteration value of the prototype from above within 15 %
        lam = proto.lam_max(fine["A"], fine["dinv"])
        assert 0.9 * 1.1 * lam <= fine["lmax"] <= 1.25 * 1.1 * lam
    cx = sum(l["A"].nnz for l in levels) / levels[0]["A"].nnz
    assert cx < 1.8
    b = np.random.default_rng(1).uniform(-1, 1, A.shape[0]) * (~bc)
    _, k_amg = proto.pcg(A, b, lambda r: proto.vcycle(levels, 0, r), 1e-5, 100)
    dinv = 1.0 / A.diagonal()
    _, k_jac = proto.pcg(A, b, lambda r: dinv * r, 1e-5, 2000)
    assert k_amg <= 8 and k_amg * 4 < k_jac, (k_amg, k_jac)


def test_setup_rejects_bad_input():
    ip = np.array([0, 1, 2], dtype=np.int32)
    ix = np.array([0, 5], dtype=np.int32)          # column out of range
    v = np.array([1.0, 1.0])
    h = ctypes.c_void_p()
    assert lib.pmgx_amg_setup_h(2, ptr(ip), ptr(ix), ptr(v), 10, 4, ctypes.addressof(h)) != 0
    ix = np.array([0, 1], dtype=np.int32)
    v = np.array([1.0, -2.0])                      # non-positive diagonal
    assert lib.pmgx_amg_setup_h(2, ptr(ip), ptr(ix), ptr(v), 0, 4, ctypes.addressof(h)) != 0


def test_setup_degenerate_sizes():
    """1 x 1, the identity (every row a Dirichlet row) and a Laplacian with identity rows appended: the set-up
    returns a hierarchy (a single level where there is nothing to coarsen) instead of failing."""
    import scipy.sparse as sp
    T = sp.diags([-1.0, 2.0, -1.0], [-1, 0, 1], shape=(100, 100))
    for A, min_levels in ((sp.eye(1) * 2.0, 1), (sp.eye(50), 1), (sp.block_diag([T, sp.eye(30)]), 2)):
        A = sp.csr_matrix(A)
        A.sort_indices()
        ip, ix = A.indptr.astype(np.int32), A.indices.astype(np.int32)
        h = ctypes.c_void_p()
        check(lib.pmgx_amg_setup_h(A.shape[0], ptr(ip), ptr(ix), ptr(A.data), 4, 10, ctypes.addressof(h)))
        assert lib.pmgx_amg_num_levels(h) >= min_levels
        lib.pmgx_amg_destroy(h)


def test_drop_stored_zeros():
    """pmgx_csr_drop_zeros_h: what the AMG coarse solver streams instead of the assembled pattern -- equal to scipy's
    eliminate_zeros except that a zero DIAGONAL entry stays; row order and entry order are preserved."""
    import scipy.sparse as sp
    rng = np.random.default_rng(11)
    n = 200
    A = sp.random(n, n, density=0.05, random_state=3, format="lil")
    A.setdiag(rng.uniform(1, 2, n))
    A = sp.csr_matrix(A)
    A.sort_indices()
    zero = rng.random(A.nnz) < 0.6
    A.data[zero] = 0.0                                    # explicit zeros, some of them on the diagonal
    ip, ix = A.indptr.astype(np.int32), A.indices.astype(np.int32)
    kept = ctypes.c_longlong(0)
    check(lib.pmgx_csr_drop_zeros_h(n, ptr(ip), ptr(ix), ptr(A.data), None, None, None, ctypes.addressof(kept)))
    rows = np.repeat(np.arange(n), np.diff(ip))
    keep = (A.data != 0.0) | (ix == rows)
    assert kept.value == int(keep.sum()) < A.nnz
    op, oc, ov = np.zeros(n + 1, np.int32), np.zeros(kept.value, np.int32), np.zeros(kept.value)
    check(lib.pmgx_csr_drop_zeros_h(n, ptr(ip), ptr(ix), ptr(A.data), ptr(op), ptr(oc), ptr(ov), ctypes.addressof(kept)))
    assert np.array_equal(op, np.concatenate([[0], np.cumsum(np.bincount(rows[keep], minlength=n))]))
    assert np.array_equal(oc, ix[keep]) and np.array_equal(ov, A.data[keep])
    B = sp.csr_matrix((ov, oc, op), shape=(n, n))
    x = rng.uniform(-1, 1, n)
    assert np.array_equal(B @ x, A @ x) or np.allclose(B @ x, A @ x, rtol=1e-15, atol=0)
    assert np.all(B.diagonal() == A.diagonal()) and all(i in oc[op[i]:op[i + 1]] for i in range(n))
    # an empty matrix
    z = np.zeros(1, np.int32)
    check(lib.pmgx_csr_drop_zeros_h(0, ptr(z), None, None, None, None, None, ctypes.addressof(kept)))
    assert kept.value == 0
