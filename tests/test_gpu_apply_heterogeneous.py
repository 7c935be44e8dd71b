"""GPU parity of the apply kernels on per-cell affine geometry, per-cell kappa and permuted cell lists, at sizes where
every persistent CTA walks over several batches.

The box is graded along each axis by a different exponential map and then sheared, so every cell is a
parallelepiped with its own geometry 6-vector Gc (all six components non-zero), and the kernels' double-buffered
dofmap, their batch rotation and their Gc / kappa indexing are exercised with data that differs from cell to cell.
kappa is random per cell and the launch order is a random permutation of the cells, so a kernel that read kappa or Gc
of the wrong cell fails here.  The reference is the C oracle (oracle/cport) on the same dofmap, BC marker and kappa.
"""
import numpy as np
import pytest
import torch

from oracle import cport, operator as oo
from helpers import rel
from test_gpu_operator import KERNELS

pytestmark = pytest.mark.gpu
TOL = 1e-12
STREAM = 4  # PMGX_LAP_STREAM_G

# Shear and offset of test_affine_geometry_kernel_on_a_sheared_box
SHEAR = np.array([[1.0, 0.3, -0.2], [0.1, 0.9, 0.25], [-0.15, 0.2, 1.1]])
OFFSET = np.array([0.3, -1.0, 2.0])
GRADING = (1.5, -2.0, 0.8)  # gamma per axis of x -> (exp(gamma x) - 1) / (exp(gamma) - 1)

# Sizes.  Every resident CTA (slab kernels) or warp (mma kernels) of the interior-cell launch must process >= 3
# batches / cells, so the double-buffered dofmap, the G ring and the batch rotation wrap several times.  A persistent
# kernel launches min(batches, CTAs per SM x SMs) CTAs; CTAs per SM is bounded from above by the thread limit
# (2048 / tpb) and the register file (65536 / (registers x tpb)), so a list of
#     count >= 3 x cpb x bound x SMs
# cells gives every CTA >= 3 batches.  Per degree: (tpb, cpb, registers per thread from `-Xptxas -v` of nvcc 12.9
# for sm_100a) of the affine kernel and of the streamed-G kernel of ApplyKernels<P>:
#   P1 k_apply_affine<1,128>       128, 64,  78 -> <= 6 CTAs | k_apply_tma<1,64>  64, 32,  80 -> <= 12
#   P2 k_apply_affine_shfl<2,128>  128, 40,  80 -> <= 6      | k_apply_tma<2,128> 128, 42, 114 -> <= 4
#   P3 k_apply_affine2<3,64>        64, 16, 158 -> <= 6      | k_apply_tma<3,128> 128, 32, 154 -> <= 3
#   P4 k_apply_affine<4,64>         64, 12, 255 -> <= 4      | k_apply_tma<4,128> 128, 25, 198 -> <= 2
#   P5 k_apply_affine<5,64>         64, 10, 255 -> <= 4      | k_apply_tma<5,64>   64, 10, 254 -> <= 4
#   P6/P7 k_apply_affine_mma        64 (2 warps, one cell per warp: cpb 2), 168 -> <= 6 CTAs (12 warps)
# P8 (k_apply<8>, 256 threads, 3 cells per CTA, 170 registers -> 1 CTA per SM) is not persistent: its list must fill
# >= 10 waves of CTAs, count >= 10 x 3 x 1 x SMs.
PERSISTENT = {
    1: [(128, 64, 78), (64, 32, 80)],
    2: [(128, 40, 80), (128, 42, 114)],
    3: [(64, 16, 158), (128, 32, 154)],
    4: [(64, 12, 255), (128, 25, 198)],
    5: [(64, 10, 255), (64, 10, 254)],
    6: [(64, 2, 168)],
    7: [(64, 2, 168)],
}
CPBS = (64, 32, 40, 42, 16, 12, 25, 10, 3)  # cells per batch of the slab kernels, cells per CTA of P8
L_SHARE = 7 / 8  # lcells take this share of the cells, bcells the rest


def _ctas_per_sm(tpb, regs):
    return min(2048 // tpb, 32, 65536 // (regs * tpb))


def _cells_needed(P, sms):
    if P == 8:
        return 10 * 3 * _ctas_per_sm(256, 170) * sms
    return max(3 * cpb * _ctas_per_sm(tpb, regs) * sms for tpb, cpb, regs in PERSISTENT[P])


def _ragged(k):
    """True when k is not a multiple of any kernel's cells per batch"""
    return all(k % c for c in CPBS)


def _size(P):
    """(n, number of lcells) of an n^3 box whose lcells list fills every resident CTA >= 3 times"""
    need = _cells_needed(P, torch.cuda.get_device_properties(0).multi_processor_count)
    n = int(np.ceil((need / L_SHARE) ** (1 / 3)))
    while True:
        nc = n ** 3
        nl = int(L_SHARE * nc)
        while not (_ragged(nl) and _ragged(nc - nl)):
            nl += 1
        if nl >= need:
            return n, nl
        n += 1


def _graded_sheared(xgeom):
    X = xgeom.copy()
    for d, g in enumerate(GRADING):
        X[:, d] = np.expm1(g * X[:, d]) / np.expm1(g)
    return X @ SHEAR.T + OFFSET


class _Case:
    """One library-generated box (graded + sheared, or perturbed), its space, per-cell kappa and permuted lists"""

    def __init__(self, ctx, P, n, nl, perturbed):
        from pmg_dolfinx_b200 import api
        m = api.BoxMesh((n, n, n), perturb=0.15 if perturbed else 0.0)
        s = m.space(P)
        self.ctx, self.P, self.nd, self.nc = ctx, P, s.n_owned, m.n_cells
        self.xgeom = m.xgeom if perturbed else _graded_sheared(m.xgeom)
        self.gdm, self.dofmap, self.bc = m.geom_dofmap, s.dofmap, s.bc
        rng = np.random.default_rng(1000 * P + perturbed)
        self.kappa = rng.uniform(0.5, 2.0, m.n_cells)
        perm = rng.permutation(m.n_cells).astype(np.int32)
        self.lcells, self.bcells = perm[:nl], perm[nl:]
        self.d = dict(kappa=ctx.to_device(self.kappa), dofmap=ctx.to_device(s.dofmap), xgeom=ctx.to_device(self.xgeom),
                      gdm=ctx.to_device(m.geom_dofmap), bc=ctx.to_device(s.bc))
        m.close()
        self.G, _ = cport.geometry(self.xgeom, self.gdm, P)

    def op(self, flags=0):
        from pmg_dolfinx_b200 import api
        d = self.d
        return api.MatFreeLaplacian(self.ctx, self.P, d["kappa"], d["dofmap"], d["xgeom"], d["gdm"], self.lcells,
                                    self.bcells, d["bc"], self.nd, 0, None, flags)

    def oracle(self, x, kappa):
        return cport.Apply(self.P, self.dofmap, self.G, kappa, self.bc, self.nd)(x)

    def apply(self, op, x):
        from pmg_dolfinx_b200 import api
        xv, yv = api.Vector(self.ctx, self.nd), api.Vector(self.ctx, self.nd)
        xv.copy_from_host(x)
        yv.set(np.nan)  # the apply overwrites y
        op(xv, yv)
        return yv.data_copy()


def _check(y, yo, what):
    e2, einf = rel(y, yo)
    assert e2 < TOL and einf < TOL, (what, e2, einf)


@pytest.mark.parametrize("P", [1, 2, 3, 4, 5, 6, 7, 8])
def test_apply_on_graded_sheared_and_perturbed_boxes_at_scale(ctx, P):
    n, nl = _size(P)
    aff = _Case(ctx, P, n, nl, perturbed=False)
    G = aff.G
    assert np.abs(G[:, :, [1, 2, 4]]).min() > 0.0                     # all six components non-zero ...
    gc = G[:, 0, :] / G[0, 0, :]
    assert np.ptp(gc, axis=0).min() > 1e-2                            # ... and different from cell to cell
    op_a, op_s = aff.op(), aff.op(STREAM)
    assert op_a.is_affine() == (P != 8) and op_a.kernel_name() == KERNELS[P][0], op_a.kernel_name()
    assert not op_s.is_affine() and op_s.kernel_name() == KERNELS[P][1], op_s.kernel_name()
    per = _Case(ctx, P, n, nl, perturbed=True)
    op_p = per.op()
    assert not op_p.is_affine() and op_p.kernel_name() == KERNELS[P][1], op_p.kernel_name()

    x = np.random.default_rng(P).uniform(-1, 1, aff.nd)
    yo = aff.oracle(x, aff.kappa)
    ya, ys = aff.apply(op_a, x), aff.apply(op_s, x)
    _check(ya, yo, (P, "affine"))
    _check(ys, yo, (P, "streamed"))
    e2, einf = rel(ya, ys)
    assert e2 < 1e-13 and einf < 1e-13, (P, "affine vs streamed", e2, einf)
    xp = np.random.default_rng(P + 50).uniform(-1, 1, per.nd)
    _check(per.apply(op_p, xp), per.oracle(xp, per.kappa), (P, "perturbed"))

    # kappa is read on every apply: scale the device coefficients in place by a non-uniform factor
    for case, ops, xx in ((aff, (op_a, op_s), x), (per, (op_p,), xp)):
        f = 1.0 + 0.5 * np.sin(np.arange(case.nc) * 0.37)
        case.d["kappa"].mul_(torch.from_numpy(f).to(case.d["kappa"].device))
        yo2 = case.oracle(xx, case.kappa * f)
        assert rel(yo2, case.oracle(xx, case.kappa))[0] > 1e-3
        for op in ops:
            _check(case.apply(op, xx), yo2, (P, op.kernel_name(), "kappa scaled in place"))


@pytest.mark.parametrize("P", [1, 2, 3, 4])
def test_diagonal_with_per_cell_kappa_and_permuted_lists(ctx, P):
    n, nl = _size(P)
    from pmg_dolfinx_b200 import api
    for perturbed in (False, True):
        case = _Case(ctx, P, n, nl, perturbed)
        do = oo.diagonal(P, case.dofmap, case.G, case.kappa, case.bc, case.nd)
        for flags in ((0, STREAM) if not perturbed else (0,)):
            op = case.op(flags)
            v = api.Vector(ctx, case.nd)
            op.get_diag_inverse(v)
            d = 1.0 / v.data_copy()
            assert np.abs(d - do).max() / np.abs(do).max() < 1e-13, (P, perturbed, op.kernel_name())
            assert (d[case.bc != 0] == 1.0).all()
