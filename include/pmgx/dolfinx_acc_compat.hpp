// dolfinx_acc_compat.hpp -- header-only C++ shim that re-creates the reference's class names
// and method signatures (Wells-Group/pmg-dolfinx, src/*.hpp) on top of the C ABI in pmgx.h,
// so that a driver written against the reference compiles with only the DOLFINx-specific
// set-up swapped (see INTEGRATION.md).  Every C status != 0 becomes a std::runtime_error, like
// the reference's own error paths (src/laplacian.hpp:346,479, src/vector.hpp:343, src/cg.hpp:125).
//
//   dolfinx::acc::Vector<T, Device>                 src/vector.hpp:74-325
//   dolfinx::acc::{inner_product,squared_norm,norm,axpy,scale,copy,pointwise_mult}
//                                                   src/vector.hpp:333-447
//   dolfinx::acc::MatFreeLaplacian<T>               src/laplacian.hpp:283-526
//   dolfinx::acc::MatrixOperator<T>                 src/csr.hpp:57-297
//   dolfinx::acc::Chebyshev<Vector>                 src/chebyshev.hpp:18-106
//   dolfinx::acc::CGSolver<Vector>                  src/cg.hpp:92-249
//   dolfinx::acc::MultigridPreconditioner<...>      src/pmg.hpp:14-183
//   Interpolator<T>                                 src/interpolate.hpp:93-329
//   CoarseSolverType<T>                             src/amg.hpp:10-118
//
// What replaces DOLFINx/Basix types: pmgx::IndexMap (owned/ghost sizes + forward-scatter lists,
// role of common::IndexMap + common::Scatterer) and pmgx::Element (a degree, role of
// basix::FiniteElement in the Interpolator constructor).
#pragma once

#include "../pmgx.h"

#include <array>
#include <cmath>
#include <cstdint>
#include <cuda_runtime.h>
#include <memory>
#include <span>
#include <stdexcept>
#include <string>
#include <vector>

namespace pmgx
{
inline void check(int status)
{
  if (status != PMGX_OK)
    throw std::runtime_error(pmgx_last_error_string());
}

/// One per GPU / rank.
class Context
{
public:
  Context(int device = 0, int rank = 0, int nranks = 1, const void* nccl_id = nullptr)
  {
    check(pmgx_ctx_create(device, rank, nranks, nccl_id, &_h));
  }
  ~Context() { pmgx_ctx_destroy(_h); }
  Context(const Context&) = delete;
  Context& operator=(const Context&) = delete;
  pmgx_ctx* handle() const { return _h; }
  cudaStream_t stream() const { return static_cast<cudaStream_t>(pmgx_ctx_stream(_h)); }
  void synchronize() const { check(pmgx_ctx_sync(_h)); }
  int rank() const { return pmgx_ctx_rank(_h); }
  int size() const { return pmgx_ctx_nranks(_h); }

private:
  pmgx_ctx* _h = nullptr;
};

/// Parallel layout of a vector: role of dolfinx::common::IndexMap + Scatterer (src/vector.hpp:83-95).
class IndexMap
{
public:
  IndexMap(std::shared_ptr<const Context> ctx, std::int32_t size_local, std::int32_t num_ghosts,
           std::span<const int> send_ranks = {}, std::span<const int> send_offsets = {},
           std::span<const std::int32_t> send_idx = {}, std::span<const int> recv_ranks = {},
           std::span<const int> recv_offsets = {}, std::span<const std::int32_t> recv_idx = {})
      : _ctx(ctx), _size_local(size_local), _num_ghosts(num_ghosts)
  {
    static const int zero = 0;
    check(pmgx_halo_create(ctx->handle(), size_local, num_ghosts, (int)send_ranks.size(), send_ranks.data(),
                           send_offsets.empty() ? &zero : send_offsets.data(), send_idx.data(),
                           (int)recv_ranks.size(), recv_ranks.data(),
                           recv_offsets.empty() ? &zero : recv_offsets.data(), recv_idx.data(), &_halo));
  }
  ~IndexMap() { pmgx_halo_destroy(_halo); }
  IndexMap(const IndexMap&) = delete;
  std::int32_t size_local() const { return _size_local; }
  std::int32_t num_ghosts() const { return _num_ghosts; }
  std::shared_ptr<const Context> ctx() const { return _ctx; }
  pmgx_halo* halo() const { return _halo; }

private:
  std::shared_ptr<const Context> _ctx;
  std::int32_t _size_local, _num_ghosts;
  pmgx_halo* _halo = nullptr;
};

/// Stand-in for basix::FiniteElement in Interpolator's constructor: a tensor-product GLL degree.
struct Element
{
  int _degree;
  explicit Element(int degree) : _degree(degree) {}
  int degree() const { return _degree; }
  int dim() const { return (_degree + 1) * (_degree + 1) * (_degree + 1); }
};

template <typename T>
struct DeviceArray
{
  T* p = nullptr;
  std::size_t n = 0;
  DeviceArray() = default;
  explicit DeviceArray(std::size_t count) { resize(count); }
  DeviceArray(const std::vector<T>& h) { assign(h.data(), h.size()); }
  DeviceArray(const DeviceArray&) = delete;
  DeviceArray& operator=(const DeviceArray&) = delete;
  DeviceArray(DeviceArray&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr, o.n = 0; }
  ~DeviceArray() { cudaFree(p); }
  void resize(std::size_t count)
  {
    cudaFree(p);
    p = nullptr;
    n = count;
    if (count && cudaMalloc(&p, count * sizeof(T)) != cudaSuccess)
      throw std::runtime_error("cudaMalloc failed");
  }
  void assign(const T* h, std::size_t count)
  {
    resize(count);
    if (count && cudaMemcpy(p, h, count * sizeof(T), cudaMemcpyHostToDevice) != cudaSuccess)
      throw std::runtime_error("cudaMemcpy failed");
  }
  std::span<const T> span() const { return {p, n}; }
};
} // namespace pmgx

namespace dolfinx::la
{
enum class Norm
{
  l2,
  linf
};
}

namespace dolfinx::acc
{
enum class Device
{
  CUDA,
  HIP,
  CPP
};

/// Distributed vector (src/vector.hpp:74-325): owned entries first, ghosts after.
template <typename T, Device D = Device::CUDA>
class Vector
{
  static_assert(std::is_same_v<T, double>, "pmgx is FP64 only");

public:
  using value_type = T;
  constexpr static Device device = D;

  Vector(std::shared_ptr<const pmgx::IndexMap> map, int bs) : _map(map), _bs(bs)
  {
    if (bs != 1)
      throw std::runtime_error("pmgx: block size must be 1");
    _n = (std::size_t)map->size_local() + map->num_ghosts();
    if (_n && cudaMalloc(&_x, _n * sizeof(T)) != cudaSuccess)
      throw std::runtime_error("cudaMalloc failed");
    set(T(0));
  }
  ~Vector() { cudaFree(_x); }
  Vector(const Vector&) = delete;
  Vector& operator=(const Vector&) = delete;

  void set(T v) { pmgx::check(pmgx_vec_set(ctx(), _x, (long long)_n, v)); }                  // :109
  template <typename HostVector>
  void copy_from_host(const HostVector& other)                                                 // :118-122
  {
    _map->ctx()->synchronize();
    cudaMemcpy(_x, other.data(), sizeof(T) * _map->size_local(), cudaMemcpyHostToDevice);
  }
  std::shared_ptr<const pmgx::IndexMap> map() const { return _map; }
  constexpr int bs() const { return _bs; }
  std::span<const T> array() const { return {_x, _n}; }
  std::span<T> mutable_array() { return {_x, _n}; }
  void scatter_fwd_begin() { pmgx::check(pmgx_halo_fwd_begin(_map->halo(), _x)); }          // :186-207
  void scatter_fwd_end() { pmgx::check(pmgx_halo_fwd_end(_map->halo(), _x)); }              // :209-238
  void scatter_fwd() { scatter_fwd_begin(), scatter_fwd_end(); }
  void scatter_rev() { pmgx::check(pmgx_halo_rev(_map->halo(), _x)); }                      // :290-294
  std::vector<T> data_copy() const                                                            // :297-302
  {
    _map->ctx()->synchronize();
    std::vector<T> h(_n);
    cudaMemcpy(h.data(), _x, _n * sizeof(T), cudaMemcpyDeviceToHost);
    return h;
  }
  pmgx_ctx* ctx() const { return _map->ctx()->handle(); }

private:
  std::shared_ptr<const pmgx::IndexMap> _map;
  int _bs;
  T* _x = nullptr;
  std::size_t _n = 0;
};

template <typename Vector>
auto inner_product(const Vector& a, const Vector& b)                                           // :333-352
{
  if (a.map()->size_local() != b.map()->size_local())
    throw std::runtime_error("Incompatible vector sizes");
  double r = 0;
  pmgx::check(pmgx_vec_dot(a.ctx(), a.array().data(), b.array().data(), a.map()->size_local(), &r));
  return r;
}
template <typename Vector>
auto squared_norm(const Vector& a) { return inner_product(a, a); }                             // :356-362
template <typename Vector>
auto norm(const Vector& a, dolfinx::la::Norm type = dolfinx::la::Norm::l2)                     // :368-390
{
  double r = 0;
  pmgx::check(pmgx_vec_norm(a.ctx(), a.array().data(), a.map()->size_local(), type == dolfinx::la::Norm::linf, &r));
  return r;
}
template <typename Vector, typename S>
void axpy(Vector& r, S alpha, const Vector& x, const Vector& y)                                 // :397-407
{
  pmgx::check(pmgx_vec_axpy(r.ctx(), r.mutable_array().data(), (double)alpha, x.array().data(), y.array().data(),
                            x.map()->size_local()));
}
template <typename Vector, typename S>
void scale(Vector& r, S alpha)                                                                  // :412-418
{
  pmgx::check(pmgx_vec_scale(r.ctx(), r.mutable_array().data(), (double)alpha, (long long)r.array().size()));
}
template <typename Vector>
void copy(Vector& a, const Vector& b)                                                           // :423-431
{
  pmgx::check(pmgx_vec_copy(a.ctx(), a.mutable_array().data(), b.array().data(), a.map()->size_local()));
}
template <typename Vector>
void pointwise_mult(Vector& w, const Vector& x, const Vector& y)                                // :437-447
{
  pmgx::check(pmgx_vec_pointwise_mult(w.ctx(), w.mutable_array().data(), x.array().data(), y.array().data(),
                                      x.map()->size_local()));
}

/// Base of the two operator flavours: owns the C handle (created lazily from the first vector's
/// map, because the reference constructors do not receive the layout either).
class OperatorBase
{
public:
  virtual ~OperatorBase() { pmgx_operator_destroy(_op); }
  template <typename Vector>
  void operator()(Vector& in, Vector& out)
  {
    ensure(in.map());
    pmgx::check(pmgx_operator_apply(_op, in.mutable_array().data(), out.mutable_array().data()));
  }
  template <typename Vector>
  void get_diag_inverse(Vector& diag_inv)
  {
    ensure(diag_inv.map());
    pmgx::check(pmgx_operator_get_diag_inverse(_op, diag_inv.mutable_array().data()));
  }
  template <typename Vector>
  void set_diag_inverse(const Vector& diag_inv)
  {
    ensure(diag_inv.map());
    pmgx::check(pmgx_operator_set_diag_inverse(_op, diag_inv.array().data()));
  }
  pmgx_operator* handle(std::shared_ptr<const pmgx::IndexMap> map)
  {
    ensure(map);
    return _op;
  }

protected:
  virtual void create(std::shared_ptr<const pmgx::IndexMap> map) = 0;
  void ensure(std::shared_ptr<const pmgx::IndexMap> map)
  {
    if (!_op)
    {
      _map = map;
      create(map);
    }
  }
  pmgx_operator* _op = nullptr;
  std::shared_ptr<const pmgx::IndexMap> _map;
};

/// Matrix-free Laplacian (src/laplacian.hpp:283-526): same constructor arguments.  The geometry
/// tables (dphi_geometry, G_weights) are accepted for signature compatibility and regenerated
/// internally.  batch_size = 0 precomputes the geometry factors once, as the reference does;
/// batch_size > 0 selects the reference's recompute mode (src/laplacian.hpp:383-396) through
/// PMGX_LAP_RECOMPUTE_G: the operator keeps no geometry and every apply forms it inside the kernel
/// from xgeom.  Nothing is stored per batch, so the value itself only selects the mode.
/// A geometry dofmap with 27 entries per cell is second-order geometry (PMGX_LAP_GEOM_Q2, node order
/// 9a + 3b + c; see INTEGRATION.md for the permutation from DOLFINx's); it does not combine with batch_size > 0.
template <typename T>
class MatFreeLaplacian : public OperatorBase
{
public:
  using value_type = T;
  MatFreeLaplacian(int degree, std::span<const T> coefficients, std::span<const std::int32_t> dofmap,
                   std::span<const T> xgeom, std::span<const std::int32_t> geometry_dofmap,
                   std::span<const T> /*dphi_geometry*/, std::span<const T> /*G_weights*/,
                   const std::vector<int>& lcells, const std::vector<int>& bcells,
                   std::span<const std::int8_t> bc_marker, std::size_t batch_size = 0)
      : degree(degree), cell_constants(coefficients), cell_dofmap(dofmap), xgeom(xgeom),
        geometry_dofmap(geometry_dofmap), bc_marker(bc_marker), lcells(lcells), bcells(bcells),
        flags(batch_size > 0 ? PMGX_LAP_RECOMPUTE_G : PMGX_LAP_DEFAULT)
  {
    if (degree < 1 || degree > PMGX_MAX_DEGREE)
      throw std::runtime_error("Unsupported degree");
    const std::size_t n_cells = dofmap.size() / ((degree + 1) * (degree + 1) * (degree + 1));
    if (n_cells > 0 && geometry_dofmap.size() == 27 * n_cells)
      flags |= PMGX_LAP_GEOM_Q2;
  }

protected:
  void create(std::shared_ptr<const pmgx::IndexMap> map) override
  {
    const int nd = (degree + 1) * (degree + 1) * (degree + 1);
    pmgx::check(pmgx_laplacian_create(map->ctx()->handle(), degree, (int)(cell_dofmap.size() / nd),
                                      cell_dofmap.data(), xgeom.data(), (int)(xgeom.size() / 3),
                                      geometry_dofmap.data(), cell_constants.data(), lcells.data(),
                                      (int)lcells.size(), bcells.data(), (int)bcells.size(), bc_marker.data(),
                                      map->size_local(), map->num_ghosts(), map->halo(), flags, &_op));
  }

private:
  int degree;
  std::span<const T> cell_constants;
  std::span<const std::int32_t> cell_dofmap;
  std::span<const T> xgeom;
  std::span<const std::int32_t> geometry_dofmap;
  std::span<const std::int8_t> bc_marker;
  std::vector<int> lcells, bcells;
  int flags;
};

/// Assembled CSR operator (src/csr.hpp:57-297).  The reference assembles a DOLFINx form; here
/// it is assembled from a matrix-free Laplacian on the same space (BC rows/cols zero, diagonal 1).
template <typename T>
class MatrixOperator : public OperatorBase
{
public:
  using value_type = T;
  MatrixOperator(MatFreeLaplacian<T>& a, std::shared_ptr<const pmgx::IndexMap> map)
  {
    _map = map;
    pmgx::check(pmgx_csr_from_laplacian(a.handle(map), &_op));
  }
  std::size_t nnz() { return (std::size_t)pmgx_csr_nnz(_op); }
  std::shared_ptr<const pmgx::IndexMap> column_index_map() { return _map; }
  std::shared_ptr<const pmgx::IndexMap> row_index_map() { return _map; }

protected:
  void create(std::shared_ptr<const pmgx::IndexMap>) override {}
};

/// 4th-kind Chebyshev smoother (src/chebyshev.hpp:18-106).
template <typename Vector>
class Chebyshev
{
  using T = typename Vector::value_type;

public:
  Chebyshev(std::shared_ptr<const pmgx::IndexMap> map, int /*bs*/, std::array<T, 2> eig_range) : _map(map)
  {
    pmgx::check(pmgx_cheb_create(map->ctx()->handle(), map->size_local(), map->num_ghosts(), eig_range[0],
                                 eig_range[1], &_h));
  }
  ~Chebyshev() { pmgx_cheb_destroy(_h); }
  void set_max_iterations(int max_iter)
  {
    _max_iter = max_iter;
    pmgx::check(pmgx_cheb_set_max_iterations(_h, max_iter));
  }
  template <typename Operator>
  T residual(Operator& A, Vector& x, const Vector& b)
  {
    T r = 0;
    pmgx::check(pmgx_cheb_residual(_h, A.handle(_map), x.mutable_array().data(), b.array().data(), &r));
    return r;
  }
  template <typename Operator>
  void solve(Operator& A, Vector& x, const Vector& b, bool verbose)
  {
    _history.assign(verbose ? _max_iter + 1 : 0, T(0));
    pmgx::check(pmgx_cheb_solve(_h, A.handle(_map), x.mutable_array().data(), b.array().data(),
                                verbose ? _history.data() : nullptr));
  }
  /// UNPRECONDITIONED residual norms of the last verbose solve (the reference logs them, :59-63,85-89)
  const std::vector<T>& residual_history() const { return _history; }
  pmgx_cheb* handle() const { return _h; }

private:
  std::shared_ptr<const pmgx::IndexMap> _map;
  pmgx_cheb* _h = nullptr;
  int _max_iter = 0;
  std::vector<T> _history;
};

/// Jacobi-preconditioned CG with Lanczos eigenvalue estimate (src/cg.hpp:92-249).
template <typename Vector>
class CGSolver
{
  using T = typename Vector::value_type;

public:
  CGSolver(std::shared_ptr<const pmgx::IndexMap> map, int /*bs*/) : _map(map)
  {
    pmgx::check(pmgx_cg_create(map->ctx()->handle(), map->size_local(), map->num_ghosts(), &_h));
  }
  ~CGSolver() { pmgx_cg_destroy(_h); }
  void set_max_iterations(int max_iter) { pmgx::check(pmgx_cg_set_max_iterations(_h, max_iter)); }
  void set_tolerance(double tolerance) { pmgx::check(pmgx_cg_set_tolerance(_h, tolerance)); }
  void store_coefficients(bool val) { pmgx::check(pmgx_cg_store_coefficients(_h, val)); }
  /// M^-1 = one V-cycle of a MultigridPreconditioner instead of the operator's diag^-1
  /// (src/cg.hpp:162,192); the reference only ever iterates its "preconditioner" (examples/pmg/main.cpp:362-367)
  template <typename PMG>
  void set_preconditioner(std::shared_ptr<PMG> pmg)
  {
    _pmg_keepalive = pmg;
    pmgx::check(pmgx_cg_set_preconditioner(_h, pmg ? pmg->handle() : nullptr));
  }
  std::vector<T> alphas() { return coeff(0); }
  std::vector<T> betas() { return coeff(1); }
  T residual() const
  {
    std::vector<T> r((std::size_t)pmgx_cg_num_coefficients(_h));
    pmgx::check(pmgx_cg_get_coefficients(_h, nullptr, nullptr, r.data()));
    return r.back();
  }
  std::vector<T> compute_eigenvalues()
  {
    std::vector<T> e((std::size_t)std::max(1, pmgx_cg_num_coefficients(_h)));
    pmgx::check(pmgx_cg_compute_eigenvalues(_h, e.data())); // throws "Insufficient data..." like :125
    e.resize((std::size_t)pmgx_cg_num_coefficients(_h));
    return e;
  }
  template <typename Operator>
  int solve(Operator& A, Vector& x, const Vector& b, bool /*verbose*/ = false)
  {
    int its = 0;
    pmgx::check(pmgx_cg_solve(_h, A.handle(_map), x.mutable_array().data(), b.array().data(), &its));
    return its;
  }

private:
  std::vector<T> coeff(int which)
  {
    std::vector<T> a((std::size_t)pmgx_cg_num_coefficients(_h)), b(a.size());
    pmgx::check(pmgx_cg_get_coefficients(_h, a.data(), b.data(), nullptr));
    return which == 0 ? a : b;
  }
  std::shared_ptr<const pmgx::IndexMap> _map;
  std::shared_ptr<void> _pmg_keepalive;
  pmgx_cg* _h = nullptr;
};
} // namespace dolfinx::acc

/// Matrix-free interpolator between two p-levels (src/interpolate.hpp:93-329).  Q1/Q2 elements
/// are pmgx::Element (degree) instead of basix::FiniteElement; the maps of the two spaces are
/// taken from the vectors of the first call.
template <typename T>
class Interpolator
{
public:
  Interpolator(const pmgx::Element& Q1_element, const pmgx::Element& Q2_element,
               std::span<const std::int32_t> Q1_dofmap, std::span<const std::int32_t> Q2_dofmap,
               std::span<const std::int32_t> l_cells, std::span<const std::int32_t> b_cells)
      : _p1(Q1_element.degree()), _p2(Q2_element.degree()), _dm1(Q1_dofmap), _dm2(Q2_dofmap),
        _lcells(l_cells.begin(), l_cells.end()), _bcells(b_cells.begin(), b_cells.end())
  {
    if (Q1_dofmap.size() / Q1_element.dim() != Q2_dofmap.size() / Q2_element.dim())
      throw std::runtime_error("Interpolator: dofmaps describe different numbers of cells");
  }
  ~Interpolator() { pmgx_interp_destroy(_h); }
  template <typename Vector>
  void interpolate(Vector& Q1_vector, Vector& Q2_vector)                                       // :185-239
  {
    ensure(Q1_vector.map(), Q2_vector.map());
    pmgx::check(pmgx_interp_prolong(_h, Q1_vector.mutable_array().data(), Q2_vector.mutable_array().data()));
  }
  template <typename Vector>
  void reverse_interpolate(Vector& Q2_vector, Vector& Q1_vector)                               // :245-303
  {
    ensure(Q1_vector.map(), Q2_vector.map());
    pmgx::check(pmgx_interp_restrict(_h, Q2_vector.mutable_array().data(), Q1_vector.mutable_array().data()));
  }
  pmgx_interp* handle(std::shared_ptr<const pmgx::IndexMap> m1, std::shared_ptr<const pmgx::IndexMap> m2)
  {
    ensure(m1, m2);
    return _h;
  }

private:
  void ensure(std::shared_ptr<const pmgx::IndexMap> m1, std::shared_ptr<const pmgx::IndexMap> m2)
  {
    if (_h)
      return;
    const int nd1 = (_p1 + 1) * (_p1 + 1) * (_p1 + 1);
    pmgx::check(pmgx_interp_create(m1->ctx()->handle(), _p1, _p2, (int)(_dm1.size() / nd1), _dm1.data(),
                                   _dm2.data(), m1->size_local() + m1->num_ghosts(),
                                   m2->size_local() + m2->num_ghosts(), _lcells.data(), (int)_lcells.size(),
                                   _bcells.data(), (int)_bcells.size(), m1->halo(), m2->halo(), &_h));
  }
  int _p1, _p2;
  std::span<const std::int32_t> _dm1, _dm2;
  std::vector<std::int32_t> _lcells, _bcells;
  pmgx_interp* _h = nullptr;
};

/// Coarse solver hook (src/amg.hpp:10-118: PETSc KSPCG + BoomerAMG, maxits 60, rtol 1e-5 there): PCG on
/// the assembled CSR operator (north_star item 5) preconditioned by a smoothed-aggregation V(2,2)
/// cycle (amg = true, collective over the ranks) or by Jacobi.
template <typename T>
class CoarseSolverType
{
public:
  CoarseSolverType(std::shared_ptr<dolfinx::acc::MatrixOperator<T>> A, std::shared_ptr<const pmgx::IndexMap> map,
                   int max_iterations = 60, double rtol = 1e-5, bool amg = true)
      : _A(A)
  {
    if (amg)
      pmgx::check(pmgx_coarse_create_amg(map->ctx()->handle(), A->handle(map), max_iterations, rtol, 2, 0, 0, &_h));
    else
      pmgx::check(pmgx_coarse_create(map->ctx()->handle(), A->handle(map), max_iterations, rtol, &_h));
  }
  ~CoarseSolverType() { pmgx_coarse_destroy(_h); }
  template <typename Vector>
  void solve(Vector& x, Vector& y)                                                              // :91-113
  {
    pmgx::check(pmgx_coarse_solve(_h, x.mutable_array().data(), y.array().data(), nullptr));
  }
  pmgx_coarse* handle() const { return _h; }

private:
  std::shared_ptr<dolfinx::acc::MatrixOperator<T>> _A;
  pmgx_coarse* _h = nullptr;
};

namespace dolfinx::acc
{
/// p-multigrid V-cycle (src/pmg.hpp:14-183).  Level 0 is the coarsest.  The reference takes the
/// level-0 BC marker only (:22-24); set_bc_markers() supplies the others (quirk Q9) -- without
/// it every level uses the constructor's marker, which is exact for two levels.
template <typename Vector, typename Operator, typename Solver, typename CoarseSolver, typename Interpolator>
class MultigridPreconditioner
{
  using T = typename Vector::value_type;

public:
  MultigridPreconditioner(std::vector<std::shared_ptr<const pmgx::IndexMap>> maps, int /*bs*/,
                          std::span<const std::int8_t> bc_marker)
      : _maps(maps), _bc(maps.size(), bc_marker.data())
  {
  }
  ~MultigridPreconditioner() { pmgx_vcycle_destroy(_h); }
  void set_solvers(std::vector<std::shared_ptr<Solver>>& solvers) { _solvers = solvers; }
  void set_coarse_solver(std::shared_ptr<CoarseSolver> solver) { _coarse_solver = solver; }
  void set_operators(std::vector<std::shared_ptr<Operator>>& operators) { _operators = operators; }
  void set_interpolators(std::vector<std::shared_ptr<Interpolator>>& interpolators) { _interp = interpolators; }
  void set_bc_markers(const std::vector<std::span<const std::int8_t>>& markers)
  {
    for (std::size_t i = 0; i < markers.size() && i < _bc.size(); ++i)
      _bc[i] = markers[i].data();
  }
  void set_flags(int flags) { _flags = flags; }

  // Apply M^{-1}x = y                                                                      :56-155
  void apply(const Vector& x, Vector& y, bool verbose = false)
  {
    if (!_h)
      build();
    T rnorm = 0;
    pmgx::check(pmgx_vcycle_apply(_h, x.array().data(), y.mutable_array().data(), verbose ? &rnorm : nullptr));
    if (verbose)
      _last_rnorm = rnorm;
  }
  T last_residual_norm() const { return _last_rnorm; } // "rnorm after PMG" (:146-149)
  /// C handle (built on first use) -- what CGSolver::set_preconditioner binds to
  pmgx_vcycle* handle()
  {
    if (!_h)
      build();
    return _h;
  }

private:
  void build()
  {
    const int nl = (int)_maps.size();
    std::vector<pmgx_operator*> ops(nl);
    std::vector<pmgx_cheb*> sm(nl);
    std::vector<pmgx_interp*> its(std::max(nl - 1, 1), nullptr);
    for (int i = 0; i < nl; ++i)
    {
      ops[i] = _operators[i]->handle(_maps[i]);
      sm[i] = _solvers[i]->handle();
      if (i < nl - 1)
        its[i] = _interp[i]->handle(_maps[i], _maps[i + 1]);
    }
    pmgx::check(pmgx_vcycle_create(_maps[0]->ctx()->handle(), nl, ops.data(), sm.data(), its.data(), _bc.data(),
                                   _coarse_solver ? _coarse_solver->handle() : nullptr, _flags, &_h));
  }
  std::vector<std::shared_ptr<const pmgx::IndexMap>> _maps;
  std::vector<const std::int8_t*> _bc;
  std::vector<std::shared_ptr<Interpolator>> _interp;
  std::vector<std::shared_ptr<Operator>> _operators;
  std::shared_ptr<CoarseSolver> _coarse_solver;
  std::vector<std::shared_ptr<Solver>> _solvers;
  pmgx_vcycle* _h = nullptr;
  int _flags = PMGX_VC_DEFAULT;
  T _last_rnorm = 0;
};
} // namespace dolfinx::acc
