"""GPU: every rank of a partition built on one device, against the single-domain oracle.

Every device object of the library is built for a rank layout: owned dofs first, then a ghost block, over the rank's
owned cells and its ghost layer, split into interior cells (lcells, no ghost dof) and boundary + ghost cells (bcells).
On one rank the ghost block is empty and the code that handles it never runs.  Without a halo (halo = None) the
Laplacian, its CSR form, the transfers, the lifting and the BC marker use the ghost block exactly as the caller left
it.  So here one process builds every rank of a partition on the one GPU, runs the forward scatter between the
emulated ranks itself with pmgx_pack / pmgx_unpack (the kernels of the NCCL path), gathers the owned entries of
every rank into one vector in the oracle's numbering and compares that with the oracle on the whole mesh.

Partitions: box grids (2,1,1), (2,2,1), (2,2,2); a ragged (3,2,1) grid on a (7,5,4) box; one-cell slabs (1,1,4) on
nz = 4, where every owned cell above rank 0 is a boundary cell and lcells is empty; scrambled general meshes (test_ghostmesh.py)
over 3 and 5 ranks; a general partition over 4 ranks that leaves one rank without cells; and a scrambled 27-node
sector (test_curved_geometry_cpu.py) over 3 ranks.  kappa is random per cell and found on every rank through the cell
centroid, so a kappa read through the wrong index on a ghost or boundary cell changes the result.

Not reached here: whatever needs two ranks with real transport -- the halo kernels behind a pmgx_halo, the
peer-memory all-reduce and the NCCL calls, the n_owned_f branches of the fused transfers, the distributed AMG and the
parked-sum branch of k_spmv_sell_cheb (tests/test_gpu_multi.py on hosts with several GPUs).
"""
from types import SimpleNamespace

import numpy as np
import pytest
import scipy.sparse as sp
import torch
from scipy.spatial import cKDTree

from oracle import mesh as om, operator as oo
from helpers import rel
import curved_reference as cr
from test_curved_geometry_cpu import scrambled_q2
from test_ghostmesh import scrambled_box
from test_gpu_operator import KERNELS
from test_gpu_recompute_geometry import KERNELS as RECOMPUTE_KERNELS

pytestmark = pytest.mark.gpu

# name: (kind, cells per direction, process grid or rank count, perturbation)
PARTITIONS = {
    "box2x1x1": ("box", (4, 3, 3), (2, 1, 1), 0.2),
    "box2x2x1": ("box", (4, 4, 3), (2, 2, 1), 0.0),
    "box2x2x2": ("box", (4, 4, 4), (2, 2, 2), 0.15),
    "ragged3x2x1": ("box", (7, 5, 4), (3, 2, 1), 0.0),
    "slabs1x1x4": ("box", (3, 3, 4), (1, 1, 4), 0.15),
    "general3": ("general", (4, 3, 3), 3, 0.15),
    "general5": ("general", (5, 3, 3), 5, 0.0),
    "empty-rank4": ("empty", (4, 3, 3), 4, 0.1),
    "curved3": ("q2", (3, 3, 2), 3, 0.1),
}
EMPTY_RANK = 1   # the rank of "empty-rank4" that owns no cell


def _parallelepipeds(X):
    """True when every cell of X [n_cells, 8, 3] (vertex order 4a + 2b + c) is a parallelepiped."""
    if len(X) == 0:
        return True
    e = X[:, [4, 2, 1]] - X[:, :1]
    abc = np.array([[a, b, c] for a in (0, 1) for b in (0, 1) for c in (0, 1)], dtype=float)
    pred = X[:, :1] + np.einsum("vk,ckd->cvd", abc, e)
    return np.abs(X - pred).max() <= 1e-12 * np.abs(X).max()


class Partition:
    """Host meshes of every rank, their device arrays, and the single-domain oracle mesh."""

    def __init__(self, ctx, api, kind, n, parts, perturb):
        self.ctx, self.api, self.kind, self.q2 = ctx, api, kind, kind == "q2"
        if kind == "box":
            full = api.BoxMesh(n, (1, 1, 1), 0, perturb=perturb)
            self.omesh = om.BoxMesh(tuple(n), full.xgeom.copy(), full.geom_dofmap.copy())
            full.close()
            self.meshes = [api.BoxMesh(n, parts, r, perturb=perturb) for r in range(int(np.prod(parts)))]
        else:
            if kind == "q2":
                self.omesh = cr.q2_box(*n, phi=cr.sector, perturb=perturb)
                cells, owner, coords = scrambled_q2(self.omesh, 3, parts)
            else:
                self.omesh, cells, owner, coords = scrambled_box(n, perturb, 5, parts - (kind == "empty"))
                if kind == "empty":
                    owner = np.where(owner >= EMPTY_RANK, owner + 1, owner).astype(np.int32)
            assert len(np.unique(owner)) == parts - (kind == "empty")
            self.meshes = [api.GhostLayerMesh(cells, owner, coords, r, parts) for r in range(parts)]
        onodes = self.omesh.verts[self.omesh.geom_dofmap]
        self.kappa = np.random.default_rng(len(self.meshes)).uniform(0.5, 2.0, self.omesh.ncells)
        ctree = cKDTree(onodes.mean(axis=1))
        self.ranks = []
        for gm in self.meshes:
            R = SimpleNamespace(mesh=gm, cell=np.zeros(0, dtype=np.int64))
            if gm.n_cells:
                dist, R.cell = ctree.query(gm.xgeom[gm.geom_dofmap].mean(axis=1))
                assert dist.max() < 1e-12
            assert len(gm.lcells) + len(gm.bcells) == gm.n_cells
            R.kappa_h = self.kappa[R.cell]
            R.kappa = ctx.to_device(R.kappa_h)
            R.xgeom, R.gdm = ctx.to_device(gm.xgeom), ctx.to_device(gm.geom_dofmap)
            R.affine = not self.q2 and _parallelepipeds(gm.xgeom[gm.geom_dofmap])
            self.ranks.append(R)
        if kind == "empty":
            assert self.meshes[EMPTY_RANK].n_cells == 0
        if kind == "box" and parts[2] == n[2]:
            # one-cell slabs: the interface dofs belong to the lower rank, so every owned cell above rank 0 touches a
            # ghost dof and lcells is empty there
            assert all(len(gm.lcells) == 0 for gm in self.meshes[1:])
        self.base_flags = api.LAP_GEOM_Q2 if self.q2 else 0
        self._levels = {}

    def close(self):
        for gm in self.meshes:
            gm.close()

    # ---- one degree: the oracle's arrays, every rank's space, canonical numbering and scatter plan
    def level(self, P):
        if P in self._levels:
            return self._levels[P]
        o, ctx = self.omesh, self.ctx
        L = SimpleNamespace(P=P, dm=om.dofmap(o, P), bc=om.bc_marker(o, P), nd=om.num_dofs(o, P))
        if self.q2:
            L.G, L.detJ = cr.geometry_factors(o.verts, o.geom_dofmap, P)
            L.X = cr.dof_coords(o, P)
        else:
            L.G, L.detJ = oo.geometry_factors(o.verts, o.geom_dofmap, P)
            L.X = om.dof_coords(o, P)
        tree = cKDTree(L.X)
        L.spaces, seen = [], np.zeros(L.nd, dtype=int)
        for R in self.ranks:
            S = R.mesh.space(P, want_coords=True)
            nt = S.n_owned + S.n_ghost
            if self.kind == "box":
                S.can = S.l2g
            else:
                S.can = tree.query(S.coords)[1] if nt else np.zeros(0, dtype=np.int64)
            assert S.n_global == L.nd
            assert np.abs(S.coords - L.X[S.can]).max(initial=0.0) < 1e-12
            assert np.array_equal(S.bc, L.bc[S.can])
            seen[S.can[: S.n_owned]] += 1
            S.dm, S.bc_d = ctx.to_device(S.dofmap), ctx.to_device(S.bc)
            L.spaces.append(S)
        assert (seen == 1).all()
        # forward scatter: for every rank r and source q, q's send segment for r and r's receive segment from q
        for r, S in enumerate(L.spaces):
            S.plan = []
            for kk, q in enumerate(S.recv_ranks):
                Sq = L.spaces[q]
                k = list(Sq.send_ranks).index(r)
                snd = Sq.send_idx[Sq.send_offsets[k]:Sq.send_offsets[k + 1]]
                rcv = S.recv_idx[S.recv_offsets[kk]:S.recv_offsets[kk + 1]]
                assert len(snd) == len(rcv) > 0
                S.plan.append((int(q), len(snd), ctx.to_device(snd), ctx.to_device(rcv)))
            assert sorted(S.recv_idx.tolist()) == list(range(S.n_ghost))
        L.checked_scatter = False
        self._levels[P] = L
        return L

    # ---- vectors of every rank
    def scatter(self, L, vecs):
        """The forward scatter between the emulated ranks, on the device: pmgx_pack of q's vector with q's send
        segment for r, pmgx_unpack into r's ghost block with r's receive segment from q."""
        from pmg_dolfinx_b200.capi import check, lib, ptr
        for S, v in zip(L.spaces, vecs):
            for q, m, snd, rcv in S.plan:
                buf = self.ctx.zeros(m)
                check(lib.pmgx_pack(self.ctx.h, m, ptr(snd), ptr(vecs[q]), ptr(buf)))
                check(lib.pmgx_unpack(self.ctx.h, m, ptr(rcv), ptr(buf), v.data_ptr() + 8 * S.n_owned))

    def distribute(self, L, xg, scatter=True):
        """device tensors of every rank: the owned entries of the global xg, ghosts by the forward scatter (NaN
        before it)"""
        vecs = []
        for S in L.spaces:
            v = torch.full((S.n_owned + S.n_ghost,), float("nan"), dtype=torch.float64, device=self.ctx.device)
            v[: S.n_owned] = torch.from_numpy(np.ascontiguousarray(xg[S.can[: S.n_owned]])).to(self.ctx.device)
            vecs.append(v)
        if scatter:
            self.scatter(L, vecs)
            if not L.checked_scatter:                # the plans pair up: every local vector is xg in local numbering
                self.ctx.sync()
                for S, v in zip(L.spaces, vecs):
                    assert np.array_equal(v.cpu().numpy(), xg[S.can])
                L.checked_scatter = True
        return vecs

    def gather(self, L, vecs):
        """one global vector from the owned entries of every rank; every global dof is written exactly once"""
        self.ctx.sync()
        out, count = np.zeros(L.nd), np.zeros(L.nd, dtype=int)
        for S, v in zip(L.spaces, vecs):
            t = v if isinstance(v, torch.Tensor) else v.data
            out[S.can[: S.n_owned]] = t[: S.n_owned].cpu().numpy()
            count[S.can[: S.n_owned]] += 1
        assert (count == 1).all()
        return out

    def vector(self, S, data=None):
        v = self.api.Vector(self.ctx, S.n_owned, S.n_ghost)
        if data is not None:
            v.data.copy_(data)
        return v

    # ---- device objects of every rank
    def laplacians(self, L, flags=0, interior_only=False):
        api, ops = self.api, []
        for R, S in zip(self.ranks, L.spaces):
            bcells = R.mesh.bcells[:0] if interior_only else R.mesh.bcells
            ops.append(api.MatFreeLaplacian(self.ctx, L.P, R.kappa, S.dm, R.xgeom, R.gdm, R.mesh.lcells, bcells, S.bc_d,
                                            S.n_owned, S.n_ghost, None, self.base_flags | flags))
        return ops

    def oracle_apply(self, L, x):
        return oo.apply(L.P, L.dm, L.G, self.kappa, L.bc, x)

    def local_G(self, R, P):
        gm = R.mesh
        return (cr.geometry_factors if self.q2 else oo.geometry_factors)(gm.xgeom, gm.geom_dofmap, P)[0]


@pytest.fixture(scope="module")
def partitions(ctx):
    from pmg_dolfinx_b200 import api
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = Partition(ctx, api, *PARTITIONS[name])
        return cache[name]
    yield get
    for p in cache.values():
        p.close()


def _apply_all(part, L, ops, xs):
    ys = [part.vector(S) for S in L.spaces]
    for op, S, x, y in zip(ops, L.spaces, xs, ys):
        op(part.vector(S, x), y)
    return ys


@pytest.mark.parametrize("P", range(1, 9))
@pytest.mark.parametrize("name", PARTITIONS)
def test_apply_matches_oracle(ctx, partitions, name, P):
    """Every geometry mode (stored G or one Gc per affine cell, streamed G, G recomputed per apply; 27-node geometry on
    the curved partition): the interior launch, then the boundary + ghost launch at batch offset nb_l."""
    part = partitions(name)
    api, L = part.api, part.level(P)
    modes = [0] if part.q2 else [0, api.LAP_STREAM_G, api.LAP_RECOMPUTE_G]
    rng = np.random.default_rng(P)
    for flags in modes:
        ops = part.laplacians(L, flags)
        for R, op in zip(part.ranks, ops):
            if R.mesh.n_cells == 0:
                continue
            affine = flags == 0 and R.affine and P < 8
            assert op.is_affine() == affine, (name, P, flags)
            expect = RECOMPUTE_KERNELS[P] if flags == api.LAP_RECOMPUTE_G else KERNELS[P][0 if affine else 1]
            assert op.kernel_name() == expect, (name, P, flags, op.kernel_name())
        if flags == 0 and PARTITIONS[name][3] == 0.0:
            # the unperturbed partitions run the affine kernels on every rank that has cells
            assert all(op.is_affine() == (P < 8) for R, op in zip(part.ranks, ops) if R.mesh.n_cells)
        for xg in (rng.uniform(-1, 1, L.nd), np.ones(L.nd)):
            y = part.gather(L, _apply_all(part, L, ops, part.distribute(L, xg)))
            e2, einf = rel(y, part.oracle_apply(L, xg))
            assert e2 < 1e-12 and einf < 1e-12, (name, P, flags, e2, einf)


@pytest.mark.parametrize("P", range(1, 9))
@pytest.mark.parametrize("name", PARTITIONS)
def test_interior_cells_never_read_ghosts(ctx, partitions, name, P):
    """An operator over lcells only, with NaN in the ghost block of x: its owned output is finite and equals the
    oracle's action of the same cells on the rank's own arrays (the overlapped apply starts the interior launch
    before the ghosts arrive)."""
    part = partitions(name)
    L = part.level(P)
    xg = np.random.default_rng(10 + P).uniform(-1, 1, L.nd)
    xs = part.distribute(L, xg, scatter=False)
    ys = _apply_all(part, L, part.laplacians(L, interior_only=True), xs)
    ctx.sync()
    for R, S, x, y in zip(part.ranks, L.spaces, xs, ys):
        got = y.data.cpu().numpy()[: S.n_owned]
        assert np.isfinite(got).all(), (name, P)
        yo = oo.apply_cells(P, S.dofmap, part.local_G(R, P), R.kappa_h, S.bc, x.cpu().numpy(),
                            np.zeros(S.n_owned + S.n_ghost), R.mesh.lcells)[: S.n_owned]
        assert np.isfinite(yo).all()
        assert np.abs(got - yo).max(initial=0.0) <= 1e-12 * np.abs(yo).max(initial=0.0), (name, P)


@pytest.mark.parametrize("P", range(1, 9))
@pytest.mark.parametrize("name", PARTITIONS)
def test_diagonal_matches_oracle(ctx, partitions, name, P):
    part = partitions(name)
    L = part.level(P)
    dvs = [part.vector(S) for S in L.spaces]
    for op, dv in zip(part.laplacians(L), dvs):
        op.get_diag_inverse(dv)
    d = 1.0 / part.gather(L, dvs)
    do = oo.diagonal(P, L.dm, L.G, part.kappa, L.bc, L.nd)
    assert np.abs(d - do).max() / np.abs(do).max() < 1e-13, (name, P)


@pytest.mark.parametrize("P", [1, 2, 3])
@pytest.mark.parametrize("name", PARTITIONS)
def test_csr_with_ghost_columns(ctx, partitions, name, P):
    """pmgx_csr_from_laplacian on every rank: owned rows with their ghost-column block.  Values against the oracle's
    assembled matrix; the pattern equal to the device CSR of the whole mesh on one rank (both keep the collocated
    zeros); the SpMV with scattered ghosts and the diagonal."""
    part = partitions(name)
    api, L = part.api, part.level(P)
    csrs = [op.to_csr() for op in part.laplacians(L)]
    rows, cols, vals, ghost_cols = [], [], [], 0
    for S, A in zip(L.spaces, csrs):
        assert A.n_owned == S.n_owned and A.n_ghost == S.n_ghost
        rp, co, va = A.to_host()
        assert rp[0] == 0 and rp[-1] == A.nnz()              # no stray entries past the last owned row
        assert ((co >= 0) & (co < S.n_owned + S.n_ghost)).all()
        r = np.repeat(np.arange(S.n_owned), np.diff(rp))
        g = co >= S.n_owned
        assert not (g[:-1] & ~g[1:] & (r[:-1] == r[1:])).any()   # owned columns first in every row
        ghost_cols += int(g.sum())
        rows.append(S.can[r])
        cols.append(S.can[co])
        vals.append(va)
    if sum(S.n_ghost for S in L.spaces):
        assert ghost_cols > 0
    rows, cols, vals = np.concatenate(rows), np.concatenate(cols), np.concatenate(vals)
    A = sp.csr_matrix((vals, (rows, cols)), shape=(L.nd, L.nd))
    assert A.nnz == len(vals)                                # no (row, column) pair twice
    A.sort_indices()
    Ao = oo.assemble_csr(P, L.dm, L.G, part.kappa, L.bc, L.nd)
    assert abs(A - Ao).max() <= 1e-13 * abs(Ao).max(), (name, P)
    # the pattern of the single-domain device matrix
    o = part.omesh
    keep = [ctx.to_device(a) for a in (part.kappa, L.dm, o.verts, o.geom_dofmap, L.bc)]
    cells = np.arange(o.ncells, dtype=np.int32)
    one = api.MatFreeLaplacian(ctx, P, keep[0], keep[1], keep[2], keep[3], cells, cells[:0], keep[4], L.nd,
                               flags=part.base_flags)
    rp1, co1, _ = one.to_csr().to_host()
    assert np.array_equal(A.indptr, rp1) and np.array_equal(A.indices, co1), (name, P)
    # SpMV with the ghosts scattered; the ghost entries of y are zeroed
    xg = np.random.default_rng(P).uniform(-1, 1, L.nd)
    ys = _apply_all(part, L, csrs, part.distribute(L, xg))
    yo = Ao @ xg
    assert np.abs(part.gather(L, ys) - yo).max() <= 1e-13 * np.abs(yo).max(), (name, P)
    for S, y in zip(L.spaces, ys):
        assert bool((y.data[S.n_owned:] == 0).all())
    dvs = [part.vector(S) for S in L.spaces]
    for A_, dv in zip(csrs, dvs):
        A_.get_diag_inverse(dv)
    do = Ao.diagonal()
    assert np.abs(1.0 / part.gather(L, dvs) - do).max() <= 1e-13 * np.abs(do).max(), (name, P)


PAIRS = [(1, 2), (1, 3), (2, 4), (3, 6), (4, 8), (1, 8), (5, 7)]


@pytest.mark.parametrize("Pc,Pf", PAIRS)
@pytest.mark.parametrize("name", ["box2x2x2", "general3", "empty-rank4"])
def test_transfers_match_oracle(ctx, partitions, name, Pc, Pf):
    """Interpolators over lcells / bcells with n_*_total = n_owned + n_ghost: multiplicity and unique-writer mask span
    the ghost cells."""
    part = partitions(name)
    api = part.api
    Lc, Lf = part.level(Pc), part.level(Pf)
    its = [api.Interpolator(ctx, Pc, Pf, Sc.dm, Sf.dm, Sc.n_owned + Sc.n_ghost, Sf.n_owned + Sf.n_ghost,
                            R.mesh.lcells, R.mesh.bcells) for R, Sc, Sf in zip(part.ranks, Lc.spaces, Lf.spaces)]
    rng = np.random.default_rng(10 * Pc + Pf)
    xc, xf = rng.uniform(-1, 1, Lc.nd), rng.uniform(-1, 1, Lf.nd)

    fine = [part.vector(S) for S in Lf.spaces]
    for it, S, x, f in zip(its, Lc.spaces, part.distribute(Lc, xc), fine):
        f.set(-7.5e30)
        it.interpolate(part.vector(S, x), f)
    pg = part.gather(Lf, fine)
    po = oo.prolong(Pc, Pf, Lc.dm, Lf.dm, xc, Lf.nd)
    assert np.abs(pg - po).max() / np.abs(po).max() < 1e-13, (name, Pc, Pf)

    coarse = [part.vector(S) for S in Lc.spaces]
    for it, S, x, c in zip(its, Lf.spaces, part.distribute(Lf, xf), coarse):
        c.set(123.0)
        it.reverse_interpolate(part.vector(S, x), c)
    rg = part.gather(Lc, coarse)
    ro = oo.restrict(Pc, Pf, Lc.dm, Lf.dm, xf, Lc.nd)
    assert np.abs(rg - ro).max() / np.abs(ro).max() < 1e-13, (name, Pc, Pf)

    a, b = np.dot(pg, xf), np.dot(xc, rg)                     # R = P^T
    assert abs(a - b) <= 1e-12 * np.linalg.norm(pg) * np.linalg.norm(xf), (a, b)


@pytest.mark.parametrize("P", [1, 3, 4, 6])
@pytest.mark.parametrize("name", PARTITIONS)
def test_rhs_and_lifting_match_oracle(ctx, partitions, name, P):
    """assemble_rhs with g = 1.3, and assemble_rhs(f, 0) + lift with per-dof Dirichlet data scattered to the ghosts:
    owned rows next to a ghost Dirichlet dof take its g from the ghost block."""
    part = partitions(name)
    L = part.level(P)
    ops = part.laplacians(L)
    f = lambda X: 1.0 + X[:, 0] * X[:, 1] - 0.5 * X[:, 2]
    gv = np.where(L.bc != 0, 1.0 + L.X[:, 0] - 2.0 * L.X[:, 2], 7.0)
    rhs = cr.rhs_collocated if part.q2 else oo.rhs_collocated
    fl = [part.ctx.to_device(f(L.X)[S.can]) for S in L.spaces]

    bs = [part.vector(S) for S in L.spaces]
    for op, fv, b in zip(ops, fl, bs):
        op.assemble_rhs(fv, 1.3, b)
    bo = rhs(part.omesh, P, f, L.bc, g=1.3, kappa=part.kappa)
    e2, einf = rel(part.gather(L, bs), bo)
    assert e2 < 1e-12 and einf < 1e-12, (name, P, e2, einf)

    bs = [part.vector(S) for S in L.spaces]
    for op, fv, g, b in zip(ops, fl, part.distribute(L, gv), bs):
        op.assemble_rhs(fv, 0.0, b)
        op.lift(g, b)
    bo = rhs(part.omesh, P, f, L.bc, g=gv, kappa=part.kappa)
    e2, einf = rel(part.gather(L, bs), bo)
    assert e2 < 1e-12 and einf < 1e-12, (name, P, e2, einf)


@pytest.mark.parametrize("P", range(1, 9))
@pytest.mark.parametrize("name", PARTITIONS)
def test_exterior_bc_marker(ctx, partitions, name, P):
    """pmgx_bc_marker_exterior without a halo: the local facet count is exact on every owned dof (the rim of the
    ghost layer may look exterior); after the forward scatter the ghost entries are the owners' too."""
    part = partitions(name)
    api, L = part.api, part.level(P)
    marks = []
    for R, S in zip(part.ranks, L.spaces):
        gdm = api.corner_columns(R.gdm) if part.q2 else R.gdm
        m = api.exterior_bc_marker(ctx, P, gdm, S.dm, S.n_owned, S.n_ghost, None)
        ctx.sync()
        assert np.array_equal(m.cpu().numpy()[: S.n_owned], S.bc[: S.n_owned]), (name, P)
        marks.append(m.to(torch.float64))
    part.scatter(L, marks)
    ctx.sync()
    for S, m in zip(L.spaces, marks):
        assert np.array_equal(m.cpu().numpy(), S.bc.astype(np.float64)), (name, P)
