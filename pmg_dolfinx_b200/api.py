"""Python mirror of the reference's operator API on top of the C ABI (include/pmgx.h).

Class and method names follow the reference headers so tests and drivers read like the
reference's own examples:
    Vector / axpy / inner_product / norm / scale / copy / pointwise_mult   src/vector.hpp
    MatFreeLaplacian.__call__ / get_diag_inverse / set_diag_inverse        src/laplacian.hpp
    MatrixOperator                                                         src/csr.hpp
    Chebyshev, CGSolver, Interpolator, CoarseSolverType,
    MultigridPreconditioner                                                src/{chebyshev,cg,interpolate,amg,pmg}.hpp
torch is used only for device memory and stream plumbing; every operation is a call into
libpmgx.so.  No CPU fallback exists.
"""
import ctypes
import numpy as np
import torch

from .capi import lib, check, ptr, PmgxError  # noqa: F401


# pmgx_laplacian_create flags (include/pmgx.h)
LAP_DEFAULT = 0
LAP_LITERAL_DETJ = 1   # detJ expression of the reference verbatim (quirk Q17)
LAP_NO_DIAG = 2        # skip the matrix-free diagonal at create
LAP_STREAM_G = 4       # stream the per-quadrature-point G even when every cell is affine
LAP_RECOMPUTE_G = 8    # keep no geometry; every apply recomputes G from xgeom (the reference's batch_size > 0)
LAP_GEOM_Q2 = 16       # 27-node (triquadratic) geometry: geometry_dofmap [n_cells, 27], node k = 9a + 3b + c

# the 8 corner nodes of a 27-node cell, in the trilinear vertex order 4a + 2b + c
Q2_CORNERS = (0, 2, 6, 8, 18, 20, 24, 26)


def corner_columns(geometry_dofmap):
    """The 8-vertex geometry dofmap of a 27-node one (numpy array or torch tensor of shape [n_cells, 27]), e.g. for
    exterior_bc_marker."""
    g = geometry_dofmap.reshape(-1, 27)[:, list(Q2_CORNERS)]
    return g.contiguous() if isinstance(g, torch.Tensor) else np.ascontiguousarray(g)


def _np(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


class Context:
    """One per GPU / rank (pmgx_ctx_create)."""

    def __init__(self, device=0, rank=0, nranks=1, nccl_id=None):
        h = ctypes.c_void_p()
        idp = None
        if nccl_id is not None:
            self._id = (ctypes.c_char * 128).from_buffer_copy(bytes(nccl_id))
            idp = ctypes.addressof(self._id)
        check(lib.pmgx_ctx_create(device, rank, nranks, idp, ctypes.addressof(h)))
        self.h = h
        self.device = torch.device("cuda", device)
        self.rank, self.nranks = rank, nranks
        # torch ops and library kernels are ordered on the same (library-owned) stream
        self.stream = torch.cuda.ExternalStream(lib.pmgx_ctx_stream(self.h), device=self.device)
        torch.cuda.set_device(self.device)
        torch.cuda.set_stream(self.stream)

    @staticmethod
    def nccl_unique_id():
        buf = (ctypes.c_char * 128)()
        check(lib.pmgx_nccl_unique_id(ctypes.addressof(buf)))
        return bytes(buf)

    def sync(self):
        check(lib.pmgx_ctx_sync(self.h))

    def launch_count(self):
        return int(lib.pmgx_ctx_launch_count(self.h))

    def zeros(self, n, dtype=torch.float64):
        return torch.zeros(int(n), dtype=dtype, device=self.device)

    def to_device(self, a, dtype=None):
        t = torch.as_tensor(np.ascontiguousarray(a))
        if dtype is not None:
            t = t.to(dtype)
        return t.to(self.device)

    def close(self):
        if self.h:
            check(lib.pmgx_ctx_destroy(self.h))
            self.h = None


def gll_tables(degree):
    n = degree + 1
    x, w, D = np.zeros(n), np.zeros(n), np.zeros(n * n)
    check(lib.pmgx_gll_tables(degree, ptr(x), ptr(w), ptr(D)))
    return x, w, D.reshape(n, n)


def gll_interp_1d(pc, pf):
    M = np.zeros((pf + 1) * (pc + 1))
    check(lib.pmgx_gll_interp_1d(pc, pf, ptr(M)))
    return M.reshape(pf + 1, pc + 1)


def exterior_bc_marker(ctx, degree, geometry_dofmap, dofmap, n_owned, n_ghost=0, halo=None):
    """Device int8 marker of the dofs on exterior facets (examples/pmg/main.cpp:173-185), owned + ghost."""
    out = torch.zeros(int(n_owned) + int(n_ghost), dtype=torch.int8, device=ctx.device)
    n_cells = int(geometry_dofmap.numel() // 8)
    check(lib.pmgx_bc_marker_exterior(ctx.h, degree, n_cells, ptr(geometry_dofmap), ptr(dofmap), int(n_owned), int(n_ghost),
                                      halo.h if halo is not None else None, ptr(out)))
    return out


def tqli(d, e):
    d = _np(d, np.float64).copy()
    e = _np(e, np.float64).copy()
    check(lib.pmgx_tqli(ptr(d), ptr(e), len(d)))
    return d


def boxmesh_fit(ndofs_total, order):
    out = np.zeros(3, dtype=np.int32)
    check(lib.pmgx_boxmesh_fit(int(ndofs_total), order, ptr(out)))
    return tuple(int(v) for v in out)


class BoxMesh:
    """Host mesh + partition (pmgx_boxmesh_*): stand-in for create_box + ghost_layer_mesh."""

    def __init__(self, n, pgrid=(1, 1, 1), rank=0, perturb=0.0, seed=1234):
        h = ctypes.c_void_p()
        check(lib.pmgx_boxmesh_create(n[0], n[1], n[2], pgrid[0], pgrid[1], pgrid[2], rank,
                                      float(perturb), seed, ctypes.addressof(h)))
        self.h = h
        self.n, self.pgrid, self.rank = tuple(n), tuple(pgrid), rank
        s = np.zeros(5, dtype=np.int64)
        check(lib.pmgx_boxmesh_sizes(self.h, ptr(s)))
        self.n_cells, self.n_owned_cells, self.n_points, nl, nb = (int(v) for v in s)
        self.xgeom = np.zeros((self.n_points, 3))
        self.geom_dofmap = np.zeros((self.n_cells, 8), dtype=np.int32)
        check(lib.pmgx_boxmesh_geometry(self.h, ptr(self.xgeom), ptr(self.geom_dofmap)))
        self.lcells = np.zeros(nl, dtype=np.int32)
        self.bcells = np.zeros(nb, dtype=np.int32)
        check(lib.pmgx_boxmesh_cell_lists(self.h, ptr(self.lcells), ptr(self.bcells)))

    def space(self, degree, want_coords=False):
        s = np.zeros(7, dtype=np.int64)
        check(lib.pmgx_boxmesh_space_sizes(self.h, degree, ptr(s)))
        sp = HostSpace()
        sp.degree = degree
        (sp.n_owned, sp.n_ghost, nsn, nst, nrn, nrt, sp.n_global) = (int(v) for v in s)
        nd3 = (degree + 1) ** 3
        nt = sp.n_owned + sp.n_ghost
        sp.dofmap = np.zeros((self.n_cells, nd3), dtype=np.int32)
        sp.bc = np.zeros(nt, dtype=np.int8)
        sp.l2g = np.zeros(nt, dtype=np.int64)
        sp.coords = np.zeros((nt, 3)) if want_coords else None
        check(lib.pmgx_boxmesh_space(self.h, degree, ptr(sp.dofmap), ptr(sp.bc), ptr(sp.l2g),
                                     ptr(sp.coords)))
        sp.send_ranks = np.zeros(nsn, dtype=np.int32)
        sp.send_offsets = np.zeros(nsn + 1, dtype=np.int32)
        sp.send_idx = np.zeros(nst, dtype=np.int32)
        sp.recv_ranks = np.zeros(nrn, dtype=np.int32)
        sp.recv_offsets = np.zeros(nrn + 1, dtype=np.int32)
        sp.recv_idx = np.zeros(nrt, dtype=np.int32)
        check(lib.pmgx_boxmesh_halo_lists(self.h, degree, ptr(sp.send_ranks), ptr(sp.send_offsets),
                                          ptr(sp.send_idx), ptr(sp.recv_ranks), ptr(sp.recv_offsets),
                                          ptr(sp.recv_idx)))
        return sp

    def close(self):
        if self.h:
            lib.pmgx_boxmesh_destroy(self.h)
            self.h = None


class HostSpace:
    pass


class GhostLayerMesh:
    """General conforming hex mesh + partition -> this rank's arrays (pmgx_ghostmesh_*): the stand-in for
    create_mesh + ghost_layer_mesh + compute_boundary_cells + dofmaps + BC marker + Scatterer lists of
    examples/pmg/main.cpp:199-256 / src/mesh.hpp:16-143 for meshes that are not lexicographic boxes.
    Same attribute surface as BoxMesh.  ``cell_vertices`` of shape [n, 27] is a second-order mesh (node order of
    LAP_GEOM_Q2; pmgx_ghostmesh_create_q2): geom_dofmap is then [n_cells, 27], and nodes_per_cell is 27."""

    def __init__(self, cell_vertices, cell_owner, coords, rank=0, nranks=1):
        cv = _np(cell_vertices, np.int64)
        npc = 27 if cv.ndim == 2 and cv.shape[1] == 27 else 8
        cv = cv.reshape(-1, npc)
        ow = _np(cell_owner, np.int32)
        xs = _np(coords, np.float64).reshape(-1, 3)
        h = ctypes.c_void_p()
        create = lib.pmgx_ghostmesh_create_q2 if npc == 27 else lib.pmgx_ghostmesh_create
        check(create(rank, nranks, len(cv), ptr(cv), ptr(ow), len(xs), ptr(xs), ctypes.addressof(h)))
        self.h, self.rank, self.nranks = h, rank, nranks
        self.nodes_per_cell = int(lib.pmgx_ghostmesh_nodes_per_cell(self.h))
        s = np.zeros(5, dtype=np.int64)
        check(lib.pmgx_ghostmesh_sizes(self.h, ptr(s)))
        self.n_cells, self.n_owned_cells, self.n_points, nl, nb = (int(v) for v in s)
        self.xgeom = np.zeros((self.n_points, 3))
        self.geom_dofmap = np.zeros((self.n_cells, self.nodes_per_cell), dtype=np.int32)
        self.cell_gid = np.zeros(self.n_cells, dtype=np.int64)
        check(lib.pmgx_ghostmesh_geometry(self.h, ptr(self.xgeom), ptr(self.geom_dofmap), ptr(self.cell_gid)))
        self.lcells = np.zeros(nl, dtype=np.int32)
        self.bcells = np.zeros(nb, dtype=np.int32)
        check(lib.pmgx_ghostmesh_cell_lists(self.h, ptr(self.lcells), ptr(self.bcells)))

    def space(self, degree, want_coords=True):
        s = np.zeros(7, dtype=np.int64)
        check(lib.pmgx_ghostmesh_space_sizes(self.h, degree, ptr(s)))
        sp = HostSpace()
        sp.degree = degree
        (sp.n_owned, sp.n_ghost, nsn, nst, nrn, nrt, sp.n_global) = (int(v) for v in s)
        nt = sp.n_owned + sp.n_ghost
        sp.dofmap = np.zeros((self.n_cells, (degree + 1) ** 3), dtype=np.int32)
        sp.bc = np.zeros(nt, dtype=np.int8)
        sp.l2g = np.zeros(nt, dtype=np.int64)
        sp.coords = np.zeros((nt, 3)) if want_coords else None
        check(lib.pmgx_ghostmesh_space(self.h, degree, ptr(sp.dofmap), ptr(sp.bc), ptr(sp.l2g), ptr(sp.coords)))
        sp.send_ranks = np.zeros(nsn, dtype=np.int32)
        sp.send_offsets = np.zeros(nsn + 1, dtype=np.int32)
        sp.send_idx = np.zeros(nst, dtype=np.int32)
        sp.recv_ranks = np.zeros(nrn, dtype=np.int32)
        sp.recv_offsets = np.zeros(nrn + 1, dtype=np.int32)
        sp.recv_idx = np.zeros(nrt, dtype=np.int32)
        check(lib.pmgx_ghostmesh_halo_lists(self.h, degree, ptr(sp.send_ranks), ptr(sp.send_offsets), ptr(sp.send_idx),
                                            ptr(sp.recv_ranks), ptr(sp.recv_offsets), ptr(sp.recv_idx)))
        return sp

    def close(self):
        if self.h:
            lib.pmgx_ghostmesh_destroy(self.h)
            self.h = None


class Halo:
    """Forward-scatter plan = IndexMap + Scatterer of a reference Vector (src/vector.hpp:83-95)."""

    def __init__(self, ctx, n_owned, n_ghost, send_ranks=(), send_offsets=(0,), send_idx=(),
                 recv_ranks=(), recv_offsets=(0,), recv_idx=()):
        self.ctx, self.n_owned, self.n_ghost = ctx, int(n_owned), int(n_ghost)
        sr, so, si = _np(send_ranks, np.int32), _np(send_offsets, np.int32), _np(send_idx, np.int32)
        rr, ro, ri = _np(recv_ranks, np.int32), _np(recv_offsets, np.int32), _np(recv_idx, np.int32)
        h = ctypes.c_void_p()
        check(lib.pmgx_halo_create(ctx.h, self.n_owned, self.n_ghost, len(sr), ptr(sr), ptr(so), ptr(si),
                                   len(rr), ptr(rr), ptr(ro), ptr(ri), ctypes.addressof(h)))
        self.h = h

    @classmethod
    def from_space(cls, ctx, sp):
        return cls(ctx, sp.n_owned, sp.n_ghost, sp.send_ranks, sp.send_offsets, sp.send_idx,
                   sp.recv_ranks, sp.recv_offsets, sp.recv_idx)


class Vector:
    """acc::Vector<T, Device::CUDA> (src/vector.hpp:74-325): owned entries then ghosts."""

    def __init__(self, ctx, n_owned, n_ghost=0, halo=None):
        self.ctx, self.n_owned, self.n_ghost, self.halo = ctx, int(n_owned), int(n_ghost), halo
        self.data = ctx.zeros(self.n_owned + self.n_ghost)

    @property
    def size_local(self):
        return self.n_owned

    def set(self, v):                                     # :109-115 (incl. ghosts)
        check(lib.pmgx_vec_set(self.ctx.h, ptr(self.data), self.n_owned + self.n_ghost, float(v)))

    def copy_from_host(self, a):                          # :118-122 (owned part only)
        a = _np(a, np.float64)
        self.data[: self.n_owned].copy_(torch.from_numpy(a[: self.n_owned]))

    def array(self):
        return self.data

    def mutable_array(self):
        return self.data

    def data_copy(self):                                  # :297-302
        self.ctx.sync()
        return self.data.cpu().numpy()

    def scatter_fwd_begin(self):                          # :186-207
        if self.halo is not None:
            check(lib.pmgx_halo_fwd_begin(self.halo.h, ptr(self.data)))

    def scatter_fwd_end(self):                            # :209-238
        if self.halo is not None:
            check(lib.pmgx_halo_fwd_end(self.halo.h, ptr(self.data)))

    def scatter_fwd(self):                                # :242-246
        self.scatter_fwd_begin()
        self.scatter_fwd_end()

    def scatter_rev(self):                                # :290-294
        if self.halo is not None:
            check(lib.pmgx_halo_rev(self.halo.h, ptr(self.data)))


def _same(a, b):
    if a.n_owned != b.n_owned:
        raise PmgxError(1, "Incompatible vector sizes")   # src/vector.hpp:342-343


def inner_product(a, b):                                  # :333-352
    _same(a, b)
    r = ctypes.c_double()
    check(lib.pmgx_vec_dot(a.ctx.h, ptr(a.data), ptr(b.data), a.n_owned, ctypes.addressof(r)))
    return r.value


def squared_norm(a):                                      # :356-362
    return inner_product(a, a)


def norm(a, kind="l2"):                                   # :368-390
    if kind not in ("l2", "linf"):
        raise PmgxError(1, "Norm type not supported")
    r = ctypes.c_double()
    check(lib.pmgx_vec_norm(a.ctx.h, ptr(a.data), a.n_owned, 1 if kind == "linf" else 0, ctypes.addressof(r)))
    return r.value


def axpy(r, alpha, x, y):                                 # :397-407  r = alpha*x + y
    check(lib.pmgx_vec_axpy(r.ctx.h, ptr(r.data), float(alpha), ptr(x.data), ptr(y.data), x.n_owned))


def scale(r, alpha):                                      # :412-418 (incl. ghosts)
    check(lib.pmgx_vec_scale(r.ctx.h, ptr(r.data), float(alpha), r.n_owned + r.n_ghost))


def copy(a, b):                                           # :423-431  a = b
    check(lib.pmgx_vec_copy(a.ctx.h, ptr(a.data), ptr(b.data), a.n_owned))


def pointwise_mult(w, x, y):                              # :437-447
    check(lib.pmgx_vec_pointwise_mult(w.ctx.h, ptr(w.data), ptr(x.data), ptr(y.data), x.n_owned))


class _Operator:
    h = None

    def __call__(self, x, y):
        check(lib.pmgx_operator_apply(self.h, ptr(x.data), ptr(y.data)))

    def get_diag_inverse(self, v):
        check(lib.pmgx_operator_get_diag_inverse(self.h, ptr(v.data)))

    def set_diag_inverse(self, v):
        check(lib.pmgx_operator_set_diag_inverse(self.h, ptr(v.data)))

    @property
    def n_owned(self):
        return lib.pmgx_operator_n_owned(self.h)

    @property
    def n_ghost(self):
        return lib.pmgx_operator_n_ghost(self.h)

    def destroy(self):
        if self.h:
            check(lib.pmgx_operator_destroy(self.h))
            self.h = None


class MatFreeLaplacian(_Operator):
    """acc::MatFreeLaplacian<T> (src/laplacian.hpp:283-526). Device tensors are borrowed."""

    def __init__(self, ctx, degree, coefficients, dofmap, xgeom, geometry_dofmap, lcells, bcells,
                 bc_marker, n_owned, n_ghost=0, halo=None, flags=0):
        self.ctx, self.degree = ctx, degree
        self._keep = (coefficients, dofmap, xgeom, geometry_dofmap, bc_marker, halo)
        lc, bc_ = _np(lcells, np.int32), _np(bcells, np.int32)
        n_cells = int(dofmap.numel() // ((degree + 1) ** 3)) if degree >= 0 else 0
        h = ctypes.c_void_p()
        check(lib.pmgx_laplacian_create(
            ctx.h, degree, n_cells, ptr(dofmap), ptr(xgeom), int(xgeom.numel() // 3), ptr(geometry_dofmap),
            ptr(coefficients), ptr(lc), len(lc), ptr(bc_), len(bc_), ptr(bc_marker), int(n_owned),
            int(n_ghost), halo.h if halo is not None else None, flags, ctypes.addressof(h)))
        self.h = h
        self.n_list = len(lc) + len(bc_)

    def is_affine(self):
        """True when the apply runs the affine-geometry kernel (one geometry 6-vector per cell)."""
        return bool(lib.pmgx_laplacian_is_affine(self.h))

    def device_bytes(self):
        """Bytes of device memory the operator owns (permutation, encoded dofmap, G, Gc, inverse diagonal)."""
        b = ctypes.c_longlong()
        check(lib.pmgx_laplacian_device_bytes(self.h, ctypes.addressof(b)))
        return b.value

    def kernel_name(self):
        buf = ctypes.create_string_buffer(96)
        check(lib.pmgx_laplacian_kernel_name(self.h, ctypes.addressof(buf), 96))
        return buf.value.decode()

    def geometry_factors(self):
        nq = (self.degree + 1) ** 3
        G = self.ctx.zeros(self.n_list * nq * 6)
        check(lib.pmgx_laplacian_get_G(self.h, ptr(G)))
        self.ctx.sync()
        return G.cpu().numpy().reshape(self.n_list, nq, 6)

    def assemble_rhs(self, fvals, g, b):
        """assemble_vector + apply_lifting + set_bc (examples/pmg/main.cpp:289-295); g: constant BC value"""
        check(lib.pmgx_laplacian_rhs(self.h, ptr(fvals), float(g), ptr(b.data)))

    def lift(self, gvals, b):
        """b -= A_full g_bc on free rows, b = g on Dirichlet rows; gvals: device tensor (owned + ghost)"""
        check(lib.pmgx_laplacian_lift(self.h, ptr(gvals), ptr(b.data)))

    def to_csr(self):
        return MatrixOperator._from_handle(self.ctx, lambda out: lib.pmgx_csr_from_laplacian(self.h, out))


class MatrixOperator(_Operator):
    """acc::MatrixOperator<T> (src/csr.hpp:57-297) from host CSR arrays."""

    def __init__(self, ctx, row_ptr, off_diag_offset, cols, values, n_ghost=0, halo=None):
        self.ctx = ctx
        rp, od = _np(row_ptr, np.int32), _np(off_diag_offset, np.int32)
        co, va = _np(cols, np.int32), _np(values, np.float64)
        h = ctypes.c_void_p()
        check(lib.pmgx_csr_create(ctx.h, len(rp) - 1, int(n_ghost), ptr(rp), ptr(od), ptr(co), ptr(va),
                                  halo.h if halo is not None else None, ctypes.addressof(h)))
        self.h = h

    @classmethod
    def _from_handle(cls, ctx, make):
        self = cls.__new__(cls)
        self.ctx = ctx
        h = ctypes.c_void_p()
        check(make(ctypes.addressof(h)))
        self.h = h
        return self

    def nnz(self):
        return int(lib.pmgx_csr_nnz(self.h))

    def to_host(self):
        n = self.n_owned
        rp = np.zeros(n + 1, dtype=np.int32)
        co = np.zeros(self.nnz(), dtype=np.int32)
        va = np.zeros(self.nnz())
        check(lib.pmgx_csr_get(self.h, ptr(rp), ptr(co), ptr(va)))
        return rp, co, va


class Chebyshev:
    """acc::Chebyshev<Vector> (src/chebyshev.hpp:18-106)."""

    def __init__(self, ctx, n_owned, n_ghost, eig_range):
        self.ctx = ctx
        h = ctypes.c_void_p()
        check(lib.pmgx_cheb_create(ctx.h, int(n_owned), int(n_ghost), float(eig_range[0]), float(eig_range[1]),
                                   ctypes.addressof(h)))
        self.h = h
        self.max_iter = 0

    def set_max_iterations(self, n):
        self.max_iter = int(n)
        check(lib.pmgx_cheb_set_max_iterations(self.h, int(n)))

    def solve(self, A, x, b, verbose=False):
        hist = np.zeros(self.max_iter + 1) if verbose else None
        check(lib.pmgx_cheb_solve(self.h, A.h, ptr(x.data), ptr(b.data), ptr(hist)))
        return hist

    def residual(self, A, x, b):
        r = ctypes.c_double()
        check(lib.pmgx_cheb_residual(self.h, A.h, ptr(x.data), ptr(b.data), ctypes.addressof(r)))
        return r.value


class CGSolver:
    """acc::CGSolver<Vector> (src/cg.hpp:92-249)."""

    def __init__(self, ctx, n_owned, n_ghost=0):
        self.ctx = ctx
        h = ctypes.c_void_p()
        check(lib.pmgx_cg_create(ctx.h, int(n_owned), int(n_ghost), ctypes.addressof(h)))
        self.h = h

    def set_max_iterations(self, n):
        check(lib.pmgx_cg_set_max_iterations(self.h, int(n)))

    def set_tolerance(self, rtol):
        check(lib.pmgx_cg_set_tolerance(self.h, float(rtol)))

    def store_coefficients(self, on):
        check(lib.pmgx_cg_store_coefficients(self.h, 1 if on else 0))

    def set_preconditioner(self, pmg):
        """M^-1 = one V-cycle of a MultigridPreconditioner (None: back to Jacobi)."""
        if pmg is not None and pmg.h is None:
            pmg._build()
        self._pmg = pmg
        check(lib.pmgx_cg_set_preconditioner(self.h, pmg.h if pmg is not None else None))

    def solve(self, A, x, b, verbose=False):
        k = ctypes.c_int()
        check(lib.pmgx_cg_solve(self.h, A.h, ptr(x.data), ptr(b.data), ctypes.addressof(k)))
        return k.value

    def _coeffs(self):
        n = lib.pmgx_cg_num_coefficients(self.h)
        a, b, r = np.zeros(n), np.zeros(n), np.zeros(n)
        check(lib.pmgx_cg_get_coefficients(self.h, ptr(a), ptr(b), ptr(r)))
        return a, b, r

    def alphas(self):
        return self._coeffs()[0]

    def betas(self):
        return self._coeffs()[1]

    def residual(self):
        return self._coeffs()[2][-1]

    def history(self, cap=4096):
        r0, n = ctypes.c_double(), ctypes.c_int()
        h = np.zeros(cap)
        check(lib.pmgx_cg_get_history(self.h, ctypes.addressof(r0), ptr(h), ctypes.addressof(n)))
        return r0.value, h[: n.value].copy()

    def compute_eigenvalues(self):
        n = lib.pmgx_cg_num_coefficients(self.h)
        e = np.zeros(max(n, 1))
        check(lib.pmgx_cg_compute_eigenvalues(self.h, ptr(e)))
        return e[:n]


class Interpolator:
    """Interpolator<T> (src/interpolate.hpp:93-329): coarse degree Q1 -> fine degree Q2."""

    def __init__(self, ctx, degree_coarse, degree_fine, Q1_dofmap, Q2_dofmap, n_coarse_total, n_fine_total,
                 l_cells, b_cells, halo_coarse=None, halo_fine=None):
        self.ctx = ctx
        self._keep = (Q1_dofmap, Q2_dofmap, halo_coarse, halo_fine)
        lc, bc_ = _np(l_cells, np.int32), _np(b_cells, np.int32)
        n_cells = int(Q1_dofmap.numel() // ((degree_coarse + 1) ** 3))
        h = ctypes.c_void_p()
        check(lib.pmgx_interp_create(ctx.h, degree_coarse, degree_fine, n_cells, ptr(Q1_dofmap), ptr(Q2_dofmap),
                                     int(n_coarse_total), int(n_fine_total), ptr(lc), len(lc), ptr(bc_), len(bc_),
                                     halo_coarse.h if halo_coarse is not None else None,
                                     halo_fine.h if halo_fine is not None else None, ctypes.addressof(h)))
        self.h = h

    def interpolate(self, Q1_vector, Q2_vector):          # :185-239
        check(lib.pmgx_interp_prolong(self.h, ptr(Q1_vector.data), ptr(Q2_vector.data)))

    def reverse_interpolate(self, Q2_vector, Q1_vector):  # :245-303
        check(lib.pmgx_interp_restrict(self.h, ptr(Q2_vector.data), ptr(Q1_vector.data)))


class CoarseSolverType:
    """CoarseSolverType<T>::solve(x, b) (src/amg.hpp:67-113: PETSc KSPCG + BoomerAMG, maxits 60, rtol 1e-5):
    PCG on the assembled CSR operator, preconditioned by one V(nu,nu) cycle of a smoothed-aggregation
    hierarchy (amg=True, the default; collective over the ranks) or by Jacobi (amg=False)."""

    def __init__(self, ctx, A_csr, max_iter=60, rtol=1e-5, amg=True, nu=2, min_coarse=0, max_levels=0):
        self.ctx, self.A, self.amg = ctx, A_csr, bool(amg)
        h = ctypes.c_void_p()
        if amg:
            check(lib.pmgx_coarse_create_amg(ctx.h, A_csr.h, int(max_iter), float(rtol), int(nu), int(min_coarse),
                                             int(max_levels), ctypes.addressof(h)))
        else:
            check(lib.pmgx_coarse_create(ctx.h, A_csr.h, int(max_iter), float(rtol), ctypes.addressof(h)))
        self.h = h

    def solve(self, x, b):
        k = ctypes.c_int()
        check(lib.pmgx_coarse_solve(self.h, ptr(x.data), ptr(b.data), ctypes.addressof(k)))
        return k.value

    def last_iterations(self):
        return int(lib.pmgx_coarse_last_iterations(self.h))

    def last_status(self):
        """(converged, relative residual sqrt(r.M^-1 r / r0.M^-1 r0) at the last host check)"""
        c, r = ctypes.c_int(), ctypes.c_double()
        check(lib.pmgx_coarse_last_status(self.h, ctypes.addressof(c), ctypes.addressof(r)))
        return bool(c.value), r.value

    def levels(self):
        """[(owned rows, nnz(A), ghosts, dense coarsest?, nnz(P))] of the hierarchy on this rank"""
        out = []
        for l in range(lib.pmgx_coarse_num_levels(self.h)):
            v = np.zeros(5, dtype=np.int64)
            check(lib.pmgx_coarse_level_info(self.h, l, ptr(v)))
            out.append(tuple(int(t) for t in v))
        return out

    def apply_preconditioner(self, r, u):
        check(lib.pmgx_coarse_apply_preconditioner(self.h, ptr(r.data), ptr(u.data)))


class MultigridPreconditioner:
    """acc::MultigridPreconditioner (src/pmg.hpp:14-183); level 0 is the coarsest."""

    def __init__(self, ctx, bc_markers, flags=0):
        self.ctx, self.bc_markers, self.flags = ctx, list(bc_markers), flags
        self.solvers = self.operators = self.interpolators = None
        self.coarse_solver = None
        self.h = None

    def set_solvers(self, s):
        self.solvers = list(s)

    def set_coarse_solver(self, s):
        self.coarse_solver = s

    def set_operators(self, o):
        self.operators = list(o)

    def set_interpolators(self, i):
        self.interpolators = list(i)

    def _build(self):
        nl = len(self.operators)
        P = ctypes.c_void_p * nl
        ops = P(*[o.h for o in self.operators])
        sm = P(*[s.h for s in self.solvers])
        bcs = P(*[ptr(b) for b in self.bc_markers])
        its = (ctypes.c_void_p * max(nl - 1, 1))(*[i.h for i in (self.interpolators or [])])
        h = ctypes.c_void_p()
        check(lib.pmgx_vcycle_create(self.ctx.h, nl, ctypes.addressof(ops), ctypes.addressof(sm),
                                     ctypes.addressof(its), ctypes.addressof(bcs),
                                     self.coarse_solver.h if self.coarse_solver is not None else None,
                                     self.flags, ctypes.addressof(h)))
        self.h = h

    def apply(self, x, y, verbose=False):
        """One V-cycle: x = right-hand side, y = solution (updated in place)."""
        if self.h is None:
            self._build()
        r = ctypes.c_double()
        check(lib.pmgx_vcycle_apply(self.h, ptr(x.data), ptr(y.data), ctypes.addressof(r) if verbose else None))
        return r.value if verbose else None

    def diagnostics(self, cap=256):
        out, n = np.zeros(cap), ctypes.c_int()
        check(lib.pmgx_vcycle_get_diagnostics(self.h, ptr(out), cap, ctypes.addressof(n)))
        return out[: n.value].copy()
