// Host orchestration + fused vector kernels of the smoother, the Krylov solver, the coarse
// solver and the V-cycle.  Replaces acc::Chebyshev (src/chebyshev.hpp), acc::CGSolver
// (src/cg.hpp), CoarseSolverType (src/amg.hpp) and acc::MultigridPreconditioner (src/pmg.hpp).
//
// Fusion (north_star items 2 and 3): every Chebyshev iteration is one operator apply plus ONE
// vector pass (r -= q, z <- c1 z + c2 D^-1 r, x += z); every CG iteration is one apply plus
// three passes (p.y | x,r update + r.D^-1 r | p update) with alpha formed on the device, so
// the host blocks once per iteration (for the reference's convergence test, src/cg.hpp:206).
#include "common.hpp"
#include "operator.hpp"
#include "reduce.cuh"
#include "solvers.hpp"

#include <cmath>
#include <cstring>

namespace pmgx
{
namespace
{
constexpr int FT = RED_THREADS;

inline int fused_grid(pmgx_ctx* c, long long n)
{
  long long b = (n + FT * 4 - 1) / (FT * 4);
  b = std::min<long long>(b, c->max_red_blocks);
  return (int)std::max<long long>(b, 1);
}

// r = b - q ; z = (D^-1 r) * c0 ; [x += z] ; optional ||r||^2        (chebyshev.hpp:56-68,73)
template <bool NORM>
__global__ void __launch_bounds__(FT)
k_cheb_init(const double* __restrict__ b, const double* __restrict__ q, const double* __restrict__ dinv,
            double* __restrict__ r, double* __restrict__ z, double* __restrict__ x, double c0,
            bool add_x, long long n, double* partials, unsigned int* counter, double* out)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  double s = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += nth)
  {
    const double rv = q ? q[i] * (-1.0) + b[i] : b[i]; // q == nullptr: x is known to be zero
    const double zv = (rv * dinv[i]) * c0;
    r[i] = rv;
    z[i] = zv;
    if (add_x)
      x[i] = q ? zv * 1.0 + x[i] : zv;
    if (NORM)
      s = fma(rv, rv, s);
  }
  if (NORM)
  {
    double v[1] = {s};
    grid_reduce<1>(v, partials, counter, out);
  }
}

// r -= q ; z = z*c1 + c2*(D^-1 r) ; [x += z] ; optional ||r||^2     (chebyshev.hpp:76-83,73)
template <bool NORM>
__global__ void __launch_bounds__(FT)
k_cheb_step(const double* __restrict__ q, const double* __restrict__ dinv, double* __restrict__ r,
            double* __restrict__ z, double* __restrict__ x, double c1, double c2, bool add_x, int defer,
            long long n, double* partials, unsigned int* counter, double* out)
{
  // defer: the x += z of the previous pass was postponed to this one (1), and x was zero (2)
  const long long nth = (long long)gridDim.x * blockDim.x;
  double s = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += nth)
  {
    const double rv = q[i] * (-1.0) + r[i];
    const double zo = z[i];
    const double zs = zo * c1;
    const double zv = (rv * dinv[i]) * c2 + zs;
    r[i] = rv;
    z[i] = zv;
    if (add_x)
    {
      const double xo = defer == 2 ? zo : (defer == 1 ? zo * 1.0 + x[i] : x[i]);
      x[i] = zv * 1.0 + xo;
    }
    if (NORM)
      s = fma(rv, rv, s);
  }
  if (NORM)
  {
    double v[1] = {s};
    grid_reduce<1>(v, partials, counter, out);
  }
}

// Last iteration: only r -= q survives (the z update of chebyshev.hpp:80-83 is never read and
// x is not touched after the last x += z at :73); optional ||r||^2.
template <bool NORM>
__global__ void __launch_bounds__(FT)
k_cheb_last(const double* __restrict__ q, double* __restrict__ r, long long n, double* partials,
            unsigned int* counter, double* out)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  double s = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += nth)
  {
    const double rv = q[i] * (-1.0) + r[i];
    r[i] = rv;
    if (NORM)
      s = fma(rv, rv, s);
  }
  if (NORM)
  {
    double v[1] = {s};
    grid_reduce<1>(v, partials, counter, out);
  }
}

// x += z*c1 + c2*(D^-1 (r - q)): the step before a dropped last iteration -- r and z are dead
template <int DUMMY>
__global__ void __launch_bounds__(FT)
k_cheb_step_xonly(const double* __restrict__ q, const double* __restrict__ dinv, const double* __restrict__ r,
                  const double* __restrict__ z, double* __restrict__ x, double c1, double c2, int defer,
                  long long n)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += nth)
  {
    const double rv = q[i] * (-1.0) + r[i];
    const double zo = z[i];
    const double zs = zo * c1;
    const double zv = (rv * dinv[i]) * c2 + zs;
    const double xo = defer == 2 ? zo : (defer == 1 ? zo * 1.0 + x[i] : x[i]);
    x[i] = zv * 1.0 + xo;
  }
}

// r = b - y ; p = D^-1 r ; rnorm0 = p.r                               (cg.hpp:160-164)
__global__ void __launch_bounds__(FT)
k_cg_init(const double* __restrict__ b, const double* __restrict__ y, const double* __restrict__ dinv,
          double* __restrict__ r, double* __restrict__ p, long long n, double* partials,
          unsigned int* counter, double* out)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  double s = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += nth)
  {
    const double rv = y[i] * (-1.0) + b[i];
    const double pv = rv * dinv[i];
    r[i] = rv;
    p[i] = pv;
    s = fma(pv, rv, s);
  }
  double v[1] = {s};
  grid_reduce<1>(v, partials, counter, out);
}

// alpha = rnorm / (p.y) ; x += alpha p ; r -= alpha y ; y = D^-1 r ; out = r.y  (cg.hpp:182-195)
__global__ void __launch_bounds__(FT)
k_cg_update(double rnorm, const double* __restrict__ rnorm_dev, const double* __restrict__ pAp,
            const double* __restrict__ p, const double* __restrict__ dinv, double* __restrict__ x,
            double* __restrict__ r, double* __restrict__ y, long long n, double* partials,
            unsigned int* counter, double* out)
{
  if (rnorm_dev)
    rnorm = *rnorm_dev; // device-resident variant (no host round trip between iterations)
  const double alpha = rnorm / *pAp;
  const double nalpha = -alpha;
  const long long nth = (long long)gridDim.x * blockDim.x;
  double s = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += nth)
  {
    const double pv = p[i];
    x[i] = pv * alpha + x[i];
    const double rv = y[i] * nalpha + r[i];
    const double yv = rv * dinv[i];
    r[i] = rv;
    y[i] = yv;
    s = fma(rv, yv, s);
  }
  double v[1] = {s};
  grid_reduce<1>(v, partials, counter, out);
}

// ---- single-reduction (Chronopoulos-Gear) PCG for the coarse solver: per iteration ONE vector
// pass, ONE SpMV and ONE pass forming both inner products, so one all-reduce of 2 doubles.
// r = b - q (q may be null: x = 0) ; u = D^-1 r ; optionally x = 0
__global__ void __launch_bounds__(FT)
k_cgcg_init(const double* __restrict__ b, const double* __restrict__ q, const double* __restrict__ dinv,
            double* __restrict__ r, double* __restrict__ u, double* __restrict__ x, bool zero_x, long long n)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += nth)
  {
    const double rv = q ? q[i] * (-1.0) + b[i] : b[i];
    r[i] = rv;
    if (dinv) // null: u = M^-1 r comes from the multilevel preconditioner right after this pass
      u[i] = rv * dinv[i];
    if (zero_x)
      x[i] = 0.0;
  }
}

// sc_cur = {gamma = r.u, delta = w.u} of this iteration, sc_old[0] = previous gamma.
//   beta = gamma/gamma_old, alpha = gamma / (delta - beta*gamma/alpha_old)   (first: beta = 0)
//   p = u + beta p ; s = w + beta s ; x += alpha p ; r -= alpha s ; u = D^-1 r
__global__ void __launch_bounds__(FT)
k_cgcg_update(const double* __restrict__ sc_cur, const double* __restrict__ sc_old,
              const double* __restrict__ alpha_old, double* __restrict__ alpha_out,
              double* __restrict__ gamma0_out, bool first,
              const double* __restrict__ dinv, const double* __restrict__ w, double* __restrict__ p,
              double* __restrict__ s, double* __restrict__ x, double* __restrict__ r, double* __restrict__ u,
              long long n)
{
  const double gamma = sc_cur[0], delta = sc_cur[1];
  double beta = first ? 0.0 : gamma / sc_old[0];
  double alpha = first ? gamma / delta : gamma / (delta - beta * gamma / *alpha_old);
  if (!(gamma > 0.0)) // r = 0: the iterate is exact, freeze it
    alpha = 0.0, beta = 0.0;
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += nth)
  {
    const double pv = first ? u[i] : fma(beta, p[i], u[i]);
    const double sv = first ? w[i] : fma(beta, s[i], w[i]);
    p[i] = pv;
    s[i] = sv;
    x[i] = fma(alpha, pv, x[i]);
    const double rv = fma(-alpha, sv, r[i]);
    r[i] = rv;
    if (dinv)
      u[i] = rv * dinv[i];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0)
  {
    *alpha_out = alpha;
    if (first)
      gamma0_out[0] = gamma; // r0.D^-1 r0 for the relative convergence test
  }
}

// out[0] = r.u, out[1] = w.u
__global__ void __launch_bounds__(FT)
k_dot2(const double* __restrict__ r, const double* __restrict__ w, const double* __restrict__ u, long long n,
       double* partials, unsigned int* counter, double* out, const PeerReduce pr)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  double a = 0.0, b = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += nth)
  {
    const double uv = u[i];
    a = fma(r[i], uv, a);
    b = fma(w[i], uv, b);
  }
  double v[2] = {a, b};
  grid_reduce<2>(v, partials, counter, out, pr); // the last block is also the all-reduce over ranks
}

void check(const char* w) { check_launch(w); }
} // namespace
} // namespace pmgx


namespace pmgx
{

// Row-complete operators (CSR): every iteration is ONE kernel -- the SpMV with the smoother's vector update
// as its epilogue (ChebEp, operator.hpp; north_star item 2).  Same recurrence, same dead-work elimination as
// below; z ping-pongs between two buffers because the SpMV gathers the old z while the new one is written.
static void cheb_solve_fused(pmgx_cheb* s, pmgx_operator* A, double* x, const double* b, bool x_is_zero,
                             ChebResidual final_r)
{
  pmgx_ctx* c = s->ctx;
  const long long n = s->n_owned;
  const double lmax = s->eig_max;
  const size_t nt = (size_t)s->n_owned + s->n_ghost;
  if (s->z2.n != nt)
  {
    s->z2.alloc(nt);
    if (nt > 0)
      PMGX_CUDA(cudaMemsetAsync(s->z2.p, 0, nt * sizeof(double), c->stream));
  }
  double* zin = s->z.p;
  double* zout = s->z2.p;
  ChebEp e;
  e.b = b;
  e.r = s->r.p;
  e.x = x;
  e.dinv = A->diag_inv.p;
  e.scratch = s->q.p;
  e.c0 = 4.0 / (3.0 * lmax);
  if (x_is_zero)
  {
    k_cheb_init<false><<<fused_grid(c, n), FT, 0, c->stream>>>(b, nullptr, e.dinv, s->r.p, zin, x, e.c0, false, n,
                                                              c->d_partials, c->d_counter, c->d_scalars + 8);
    check("k_cheb_init");
    count_launch(c);
  }
  else
  {
    e.mode = ChebEp::INIT;
    e.z_out = zin;
    A->apply_cheb(x, e);                                                           // :56-68
  }
  const int defer_mode = x_is_zero ? 2 : 1; // max_iter >= 2: the first x += z is always formed in the next pass
  for (int i = 1; i <= s->max_iter; ++i)
  {
    const bool last = i == s->max_iter;
    if (last && final_r == CHEB_R_NONE)
      break;
    if (last && final_r == CHEB_R_SPLIT)
    {
      A->apply(zin, s->q.p); // r = s->r - s->q, combined by the caller
      break;
    }
    e.c1 = double(2 * i - 1) / double(2 * i + 3);
    e.c2 = double(8 * i + 4) / double(2 * i + 3) / lmax;
    e.defer = i == 1 ? defer_mode : 0;
    e.mode = last ? ChebEp::LAST : ((i + 1 == s->max_iter && final_r == CHEB_R_NONE) ? ChebEp::XONLY : ChebEp::STEP);
    e.z_out = zout;
    A->apply_cheb(zin, e);                                                         // :76-83 (+ :73 of the next iteration)
    if (e.mode == ChebEp::STEP)
      std::swap(zin, zout);
  }
}

void cheb_solve(pmgx_cheb* s, pmgx_operator* A, double* x, const double* b, double* hist, bool x_is_zero,
                ChebResidual final_r)
{
  if (!hist && s->max_iter >= 2 && A->supports_cheb_fusion())
    return cheb_solve_fused(s, A, x, b, x_is_zero, final_r);
  pmgx_ctx* c = s->ctx;
  const long long n = s->n_owned;
  const double lmax = s->eig_max; // only the upper bound is used (chebyshev.hpp:51)
  const double* dinv = A->diag_inv.p; // get_diag_inverse without the per-call copy (:53)
  const int grid = fused_grid(c, n);
  if (hist)
    final_r = CHEB_R_FULL; // every iteration's ||r|| is reported
  if (s->max_iter == 0 && final_r == CHEB_R_SPLIT)
    final_r = CHEB_R_FULL;
  if (!x_is_zero)
    A->apply(x, s->q.p); // :56
  const double* q0 = x_is_zero ? nullptr : s->q.p; // A*0 = 0: skip the apply, r = b
  // x += z0 (:73, first iteration) is postponed to the next pass whenever that pass updates x
  // anyway: it then forms (x + z0) + z1 in the reference's order and this pass does not touch x
  const bool deferred = s->max_iter >= 2; // then the pass of iteration 1 is never the last one
  const bool first_add = s->max_iter >= 1 && !deferred;
  const int defer_mode = !deferred ? 0 : (x_is_zero ? 2 : 1);
  const double c0 = 4.0 / (3.0 * lmax);
  if (hist)
    k_cheb_init<true><<<grid, FT, 0, c->stream>>>(b, q0, dinv, s->r.p, s->z.p, x, c0, first_add, n,
                                                  c->d_partials, c->d_counter, c->d_scalars + 8);
  else
    k_cheb_init<false><<<grid, FT, 0, c->stream>>>(b, q0, dinv, s->r.p, s->z.p, x, c0, first_add, n,
                                                   c->d_partials, c->d_counter, c->d_scalars + 8);
  check("k_cheb_init");
  count_launch(c);
  if (hist)
  {
    vec::allreduce_scalars(c, 8, 1, false);
    hist[0] = std::sqrt(vec::read_scalar(c, 8));
  }
  for (int i = 1; i <= s->max_iter; ++i)
  {
    const bool last = i == s->max_iter;
    if (last && final_r == CHEB_R_NONE)
      break; // nothing of this iteration is observable
    A->apply(s->z.p, s->q.p); // :76
    if (last && final_r == CHEB_R_SPLIT)
      break; // r = s->r - s->q, combined by the caller
    const double c1 = double(2 * i - 1) / double(2 * i + 3);
    const double c2 = double(8 * i + 4) / double(2 * i + 3) / lmax;
    if (last)
    {
      if (hist)
        k_cheb_last<true><<<grid, FT, 0, c->stream>>>(s->q.p, s->r.p, n, c->d_partials, c->d_counter,
                                                      c->d_scalars + 8);
      else
        k_cheb_last<false><<<grid, FT, 0, c->stream>>>(s->q.p, s->r.p, n, c->d_partials, c->d_counter,
                                                       c->d_scalars + 8);
      check("k_cheb_last");
    }
    else if (i + 1 == s->max_iter && final_r == CHEB_R_NONE)
    {
      // the next iteration is dropped, so r and z of this one are dead as well
      k_cheb_step_xonly<0><<<grid, FT, 0, c->stream>>>(s->q.p, dinv, s->r.p, s->z.p, x, c1, c2,
                                                       i == 1 ? defer_mode : 0, n);
      check("k_cheb_step_xonly");
    }
    else
    {
      // the x += z of iteration i+1 (:73) is folded into this pass
      if (hist)
        k_cheb_step<true><<<grid, FT, 0, c->stream>>>(s->q.p, dinv, s->r.p, s->z.p, x, c1, c2, true,
                                                      i == 1 ? defer_mode : 0, n, c->d_partials, c->d_counter,
                                                      c->d_scalars + 8);
      else
        k_cheb_step<false><<<grid, FT, 0, c->stream>>>(s->q.p, dinv, s->r.p, s->z.p, x, c1, c2, true,
                                                       i == 1 ? defer_mode : 0, n, c->d_partials, c->d_counter,
                                                       c->d_scalars + 8);
      check("k_cheb_step");
    }
    count_launch(c);
    if (hist)
    {
      vec::allreduce_scalars(c, 8, 1, false);
      hist[i] = std::sqrt(vec::read_scalar(c, 8));
    }
  }
}
} // namespace pmgx

// -------------------------------------------------------------------------------- CG --

namespace pmgx
{
// CGSolver::solve with M^-1 = one p-multigrid V-cycle from a zero initial guess
// (MultigridPreconditioner::apply, src/pmg.hpp:56-155) in the two places where src/cg.hpp:162,192
// multiply by diag^-1 -- SURVEY 8f-4: "the class is named Preconditioner but the example only
// iterates it".  Same order of operations, same break-before-store semantics (:206-218); the cycle
// costs three orders of magnitude more than the vector updates, so they are left unfused.
int cg_solve_pmg(pmgx_cg* s, pmgx_operator* A, double* x, const double* b)
{
  pmgx_ctx* c = s->ctx;
  const long long n = s->n_owned;
  const long long nt = (long long)s->n_owned + s->n_ghost;
  auto precond = [&](const double* r, double* z)
  {
    vec::set(c, z, nt, 0.0); // apply(x = r, y = z) improves z: start from zero
    const int rc = pmgx_vcycle_apply(s->precond, r, z, nullptr);
    if (rc != PMGX_OK)
      throw Error{rc};
  };
  s->history.clear();
  A->apply(x, s->y.p);                                                           // :159
  vec::axpy(c, s->r.p, -1.0, s->y.p, b, n);                                      // :160
  precond(s->r.p, s->p.p);                                                       // :162
  const double rnorm0 = vec::dot(c, s->p.p, s->r.p, n);                          // :164
  s->rnorm0 = rnorm0;
  double rnorm = rnorm0;
  const double rtol2 = s->rtol * s->rtol;
  int k = 0;
  while (k < s->max_iter)
  {
    ++k;
    A->apply(s->p.p, s->y.p);                                                    // :179
    const double alpha = rnorm / vec::dot(c, s->p.p, s->y.p, n);                 // :182
    vec::axpy(c, x, alpha, s->p.p, x, n);                                        // :186
    vec::axpy(c, s->r.p, -alpha, s->y.p, s->r.p, n);                             // :189
    precond(s->r.p, s->y.p);                                                     // :192
    const double rnorm_new = vec::dot(c, s->r.p, s->y.p, n);                     // :195
    const double beta = rnorm_new / rnorm;
    rnorm = rnorm_new;
    s->history.push_back(rnorm);
    if (rnorm / rnorm0 < rtol2)                                                  // :206
      break;
    vec::axpy(c, s->p.p, beta, s->p.p, s->y.p, n);                               // :211
    if (s->store)
    {
      s->alphas.push_back(alpha);
      s->betas.push_back(beta);
      s->residuals.push_back(rnorm);
    }
  }
  return k;
}

int cg_solve(pmgx_cg* s, pmgx_operator* A, double* x, const double* b)
{
  if (s->precond)
    return cg_solve_pmg(s, A, x, b);
  pmgx_ctx* c = s->ctx;
  const long long n = s->n_owned;
  const double* dinv = A->diag_inv.p;
  const int grid = fused_grid(c, n);
  s->history.clear();
  A->apply(x, s->y.p);                                                           // :159
  k_cg_init<<<grid, FT, 0, c->stream>>>(b, s->y.p, dinv, s->r.p, s->p.p, n, c->d_partials,
                                        c->d_counter, c->d_scalars + 1);          // :160-164
  check("k_cg_init");
  count_launch(c);
  vec::allreduce_scalars(c, 1, 1, false);
  const double rnorm0 = vec::read_scalar(c, 1);
  s->rnorm0 = rnorm0;
  double rnorm = rnorm0;
  const double rtol2 = s->rtol * s->rtol;
  int k = 0;
  while (k < s->max_iter)
  {
    ++k;
    A->apply(s->p.p, s->y.p);                                                    // :179
    vec::dot_device(c, s->p.p, s->y.p, n, 2);                                    // :182
    k_cg_update<<<grid, FT, 0, c->stream>>>(rnorm, nullptr, c->d_scalars + 2, s->p.p, dinv, x, s->r.p, s->y.p, n,
                                            c->d_partials, c->d_counter, c->d_scalars + 3); // :186-195
    check("k_cg_update");
    count_launch(c);
    vec::allreduce_scalars(c, 3, 1, false);
    // one host round trip per iteration: p.y (for alpha) and the new r.M^-1 r
    vec::publish_scalars(c, 2, 2);
    const double alpha = rnorm / c->h_scalars[2];
    const double rnorm_new = c->h_scalars[3];
    const double beta = rnorm_new / rnorm;
    rnorm = rnorm_new;
    s->history.push_back(rnorm);
    if (rnorm / rnorm0 < rtol2)                                                  // :206
      break;
    vec::axpy(c, s->p.p, beta, s->p.p, s->y.p, n);                               // :211
    if (s->store)
    {
      s->alphas.push_back(alpha);
      s->betas.push_back(beta);
      s->residuals.push_back(rnorm);
    }
  }
  return k;
}
} // namespace pmgx

namespace pmgx
{
// Coarse-level PCG, single-reduction form: mathematically the CG of src/cg.hpp, but the two inner
// products of an iteration are formed together in one pass, alpha/beta never leave the device
// and the host only looks at r.M^-1 r every `check_every` iterations.  M is the smoothed-
// aggregation V-cycle of amg.cu (the reference runs PETSc CG + BoomerAMG here, src/amg.hpp:33-47)
// or Jacobi.  Iteration counts of this inner solve are not a parity quantity.
int cgcg_solve(pmgx_coarse* co, double* x, const double* b, bool x_is_zero)
{
  pmgx_cg* s = co->cg;
  pmgx_operator* A = co->A;
  Precond* M = co->M;
  const int check_every = co->check_every;
  pmgx_ctx* c = s->ctx;
  const long long n = s->n_owned;
  const double* dinv = M ? nullptr : A->diag_inv.p;
  const int grid = fused_grid(c, n);
  const size_t nt = (size_t)s->n_owned + s->n_ghost;
  // the five work vectors live in one slab
  const size_t ntp = (nt + 15) & ~(size_t)15;
  if (s->slab.n != 5 * ntp)
  {
    s->slab.alloc(5 * ntp);
    if (nt > 0)
      PMGX_CUDA(cudaMemsetAsync(s->slab.p, 0, 5 * ntp * sizeof(double), c->stream));
    if (s->graph)
      cudaGraphExecDestroy(s->graph);
    if (s->graph_odd)
      cudaGraphExecDestroy(s->graph_odd);
    s->graph = s->graph_odd = nullptr;
  }
  double* const cr = s->slab.p;            // r
  double* const w = s->slab.p + ntp;       // w = A u
  double* const cp = s->slab.p + 2 * ntp;  // p
  double* const cu = s->slab.p + 3 * ntp;  // u = D^-1 r
  double* const cs = s->slab.p + 4 * ntp;  // s = A p
  // (An L2 access-policy window that pins this slab in a persisting set-aside was measured: the
  // coarse solve gains 4 %, but the set-aside costs the fine-level kernels their L2 and the whole
  // V-cycle goes from 22 to 31 ms -- not used.)
  double* sc = c->d_scalars + 16;  // sc[2*(it&1) + {0,1}] = {gamma, delta}
  double* al = c->d_scalars + 20;  // al[it&1] = alpha
  auto spmv_dots = [&](double* out2, int slot)
  {
    A->apply(cu, w);
    const PeerReduce pr = p2p::next_epoch(c);
    k_dot2<<<grid, FT, 0, c->stream>>>(cr, w, cu, n, c->d_partials, c->d_counter, out2, pr);
    check("k_dot2");
    count_launch(c);
    if (pr.nranks == 0)
      vec::allreduce_scalars(c, slot, 2, false); // NCCL (no-op on one rank)
  };
  if (!x_is_zero)
    A->apply(x, w);
  k_cgcg_init<<<grid, FT, 0, c->stream>>>(b, x_is_zero ? nullptr : w, dinv, cr, cu, x, x_is_zero, n);
  check("k_cgcg_init");
  count_launch(c);
  if (M)
    M->apply(cr, cu);
  spmv_dots(sc, 16);
  s->history.clear();
  const double rtol2 = s->rtol * s->rtol;
  double* g0 = c->d_scalars + 22; // gamma of iteration 0, next to the ping-pong slots: one D2H reads both
  // one full iteration: vector update with the scalars of slot k&1, then SpMV + inner products
  // into the other slot
  auto iterate = [&](int k)
  {
    const int cur = k & 1, nxt = cur ^ 1;
    k_cgcg_update<<<grid, FT, 0, c->stream>>>(sc + 2 * cur, sc + 2 * nxt, al + nxt, al + cur, g0, k == 0, dinv, w,
                                              cp, cs, x, cr, cu, n);
    check("k_cgcg_update");
    count_launch(c);
    if (k + 1 < s->max_iter)
    {
      if (M)
        M->apply(cr, cu);
      spmv_dots(sc + 2 * nxt, 16 + 2 * nxt);
    }
  };
  // blocks [k0, k0 + check_every) with k0 even, k0 >= 2 and no last iteration inside are identical
  // launch sequences: capture once, replay
  // (an odd block length alternates between two graphs, one per parity of the scalar slots)
  auto run_block = [&](int k0)
  {
    const void* key[3] = {A, x, reinterpret_cast<const void*>((size_t)check_every)};
    if ((s->graph || s->graph_odd) && (s->graph_key[0] != key[0] || s->graph_key[1] != key[1] || s->graph_key[2] != key[2]))
    {
      if (s->graph)
        cudaGraphExecDestroy(s->graph);
      if (s->graph_odd)
        cudaGraphExecDestroy(s->graph_odd);
      s->graph = s->graph_odd = nullptr;
    }
    cudaGraphExec_t& slot_graph = (k0 & 1) ? s->graph_odd : s->graph;
    if (!slot_graph)
    {
      const long long l0 = c->launches;
      cudaGraph_t g = nullptr;
      bool ok = cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeRelaxed) == cudaSuccess;
      if (ok)
      {
        try
        {
          for (int k = k0; k < k0 + check_every; ++k)
            iterate(k);
        }
        catch (const Error&)
        {
          ok = false;
        }
        ok = (cudaStreamEndCapture(c->stream, &g) == cudaSuccess) && ok && g != nullptr;
      }
      if (ok)
        ok = cudaGraphInstantiate(&slot_graph, g, 0) == cudaSuccess;
      if (g)
        cudaGraphDestroy(g);
      s->graph_launches = (int)(c->launches - l0);
      c->launches = l0;
      if (!ok)
      {
        cudaGetLastError();
        slot_graph = nullptr;
        s->graph_off = true; // this configuration cannot be captured: plain launches from now on
        for (int k = k0; k < k0 + check_every; ++k)
          iterate(k);
        return;
      }
      s->graph_key[0] = key[0], s->graph_key[1] = key[1], s->graph_key[2] = key[2];
    }
    PMGX_CUDA(cudaGraphLaunch(slot_graph, c->stream));
    count_launch(c, s->graph_launches);
  };
  int k = 0;
  co->last_converged = false;
  co->last_rel = 0.0;
  while (k < s->max_iter)
  {
    if (k >= 2 && k % check_every == 0 && k + check_every < s->max_iter && !s->graph_off)
    {
      run_block(k);
      k += check_every;
    }
    else
    {
      iterate(k);
      ++k;
      if (k == s->max_iter)
        break;
    }
    const int nxt = k & 1; // slot written by the last spmv_dots
    if (k % check_every == 0)
    {
      // the only host round trips of the solve: gamma slots 16..19, alpha 20..21, gamma0 22
      vec::publish_scalars(c, 16, 7);
      const double r = c->h_scalars[16 + 2 * nxt];
      s->rnorm0 = c->h_scalars[22];
      s->history.push_back(r);
      co->last_rel = s->rnorm0 > 0.0 ? std::sqrt(std::max(r, 0.0) / s->rnorm0) : 0.0;
      if (!(r > 0.0) || r / s->rnorm0 < rtol2)
      {
        co->last_converged = true;
        break;
      }
    }
  }
  return k;
}
} // namespace pmgx

// ------------------------------------------------------------------------ coarse solver --

// ----------------------------------------------------------------------------- V-cycle --
struct pmgx_vcycle
{
  pmgx_ctx* ctx = nullptr;
  int n_levels = 0;
  int flags = 0;
  std::vector<pmgx_operator*> ops;
  std::vector<pmgx_cheb*> smoothers;
  std::vector<pmgx_interp*> interps;
  std::vector<const int8_t*> bc;
  pmgx_coarse* coarse = nullptr;
  std::vector<pmgx::DevBuf<double>> u, r, b; // src/pmg.hpp:165-168 (du folded into the prolongation)
  std::vector<double> diagnostics;
};

extern "C"
{
// ---- Chebyshev
int pmgx_cheb_create(pmgx_ctx* ctx, int n_owned, int n_ghost, double eig_min, double eig_max, pmgx_cheb** out)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(ctx && out && n_owned >= 0 && n_ghost >= 0, "cheb_create: bad arguments");
  PMGX_REQUIRE(eig_max > 0.0, "cheb_create: eig_max must be positive");
  PMGX_CUDA(cudaSetDevice(ctx->device));
  std::unique_ptr<pmgx_cheb> s(new pmgx_cheb());
  s->ctx = ctx;
  s->n_owned = n_owned;
  s->n_ghost = n_ghost;
  s->eig_min = eig_min;
  s->eig_max = eig_max;
  const size_t nt = (size_t)n_owned + n_ghost;
  s->z.alloc(nt);
  s->q.alloc(nt);
  s->r.alloc(nt);
  if (nt > 0)
  {
    PMGX_CUDA(cudaMemsetAsync(s->z.p, 0, nt * sizeof(double), ctx->stream));
    PMGX_CUDA(cudaMemsetAsync(s->q.p, 0, nt * sizeof(double), ctx->stream));
    PMGX_CUDA(cudaMemsetAsync(s->r.p, 0, nt * sizeof(double), ctx->stream));
  }
  *out = s.release();
  PMGX_API_END
}
int pmgx_cheb_set_max_iterations(pmgx_cheb* s, int max_iter)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(s && max_iter >= 0, "cheb_set_max_iterations: bad arguments");
  s->max_iter = max_iter;
  PMGX_API_END
}
int pmgx_cheb_solve(pmgx_cheb* s, pmgx_operator* A, double* x, const double* b, double* resid_hist_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(s && A && x && b, "cheb_solve: null argument");
  PMGX_REQUIRE(A->n_owned == s->n_owned && A->n_ghost == s->n_ghost, "Incompatible vector sizes");
  PMGX_CUDA(cudaSetDevice(s->ctx->device));
  // the recurrence residual is private to the solver: drop the reference's dead last iteration
  pmgx::cheb_solve(s, A, x, b, resid_hist_h, false, pmgx::CHEB_R_NONE);
  PMGX_API_END
}
int pmgx_cheb_residual(pmgx_cheb* s, pmgx_operator* A, double* x, const double* b, double* rnorm_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(s && A && x && b && rnorm_h, "cheb_residual: null argument");
  PMGX_REQUIRE(A->n_owned == s->n_owned && A->n_ghost == s->n_ghost, "Incompatible vector sizes");
  PMGX_CUDA(cudaSetDevice(s->ctx->device));
  A->apply(x, s->q.p);                                                  // chebyshev.hpp:40
  pmgx::vec::axpy(s->ctx, s->r.p, -1.0, s->q.p, b, s->n_owned);         // :41
  *rnorm_h = std::sqrt(pmgx::vec::dot(s->ctx, s->r.p, s->r.p, s->n_owned));
  PMGX_API_END
}
int pmgx_cheb_destroy(pmgx_cheb* s)
{
  PMGX_API_BEGIN
  if (s)
  {
    cudaSetDevice(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    delete s;
  }
  PMGX_API_END
}

// ---- CG
int pmgx_cg_create(pmgx_ctx* ctx, int n_owned, int n_ghost, pmgx_cg** out)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(ctx && out && n_owned >= 0 && n_ghost >= 0, "cg_create: bad arguments");
  PMGX_CUDA(cudaSetDevice(ctx->device));
  std::unique_ptr<pmgx_cg> s(new pmgx_cg());
  s->ctx = ctx;
  s->n_owned = n_owned;
  s->n_ghost = n_ghost;
  const size_t nt = (size_t)n_owned + n_ghost;
  s->r.alloc(nt);
  s->y.alloc(nt);
  s->p.alloc(nt);
  if (nt > 0)
  {
    PMGX_CUDA(cudaMemsetAsync(s->r.p, 0, nt * sizeof(double), ctx->stream));
    PMGX_CUDA(cudaMemsetAsync(s->y.p, 0, nt * sizeof(double), ctx->stream));
    PMGX_CUDA(cudaMemsetAsync(s->p.p, 0, nt * sizeof(double), ctx->stream));
  }
  *out = s.release();
  PMGX_API_END
}
int pmgx_cg_set_max_iterations(pmgx_cg* s, int max_iter)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(s && max_iter >= 0, "cg_set_max_iterations: bad arguments");
  s->max_iter = max_iter;
  s->alphas.reserve(max_iter);
  s->betas.reserve(max_iter);
  s->residuals.reserve(max_iter);
  PMGX_API_END
}
int pmgx_cg_set_tolerance(pmgx_cg* s, double rtol)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(s, "cg_set_tolerance: null solver");
  s->rtol = rtol;
  PMGX_API_END
}
int pmgx_cg_set_preconditioner(pmgx_cg* s, pmgx_vcycle* M)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(s, "cg_set_preconditioner: null solver");
  s->precond = M;
  PMGX_API_END
}
int pmgx_cg_store_coefficients(pmgx_cg* s, int on)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(s, "cg_store_coefficients: null solver");
  s->store = on != 0;
  PMGX_API_END
}
int pmgx_cg_solve(pmgx_cg* s, pmgx_operator* A, double* x, const double* b, int* iters_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(s && A && x && b, "cg_solve: null argument");
  PMGX_REQUIRE(A->n_owned == s->n_owned && A->n_ghost == s->n_ghost, "Incompatible vector sizes");
  PMGX_CUDA(cudaSetDevice(s->ctx->device));
  const int k = pmgx::cg_solve(s, A, x, b);
  if (iters_h)
    *iters_h = k;
  PMGX_API_END
}
int pmgx_cg_num_coefficients(pmgx_cg* s) { return s ? (int)s->alphas.size() : -1; }
int pmgx_cg_get_coefficients(pmgx_cg* s, double* alphas_h, double* betas_h, double* residuals_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(s, "cg_get_coefficients: null solver");
  for (size_t i = 0; i < s->alphas.size(); ++i)
  {
    if (alphas_h)
      alphas_h[i] = s->alphas[i];
    if (betas_h)
      betas_h[i] = s->betas[i];
    if (residuals_h)
      residuals_h[i] = s->residuals[i];
  }
  PMGX_API_END
}
int pmgx_cg_get_history(pmgx_cg* s, double* rnorm0_h, double* rnorms_h, int* n_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(s, "cg_get_history: null solver");
  if (rnorm0_h)
    *rnorm0_h = s->rnorm0;
  if (n_h)
    *n_h = (int)s->history.size();
  if (rnorms_h)
    for (size_t i = 0; i < s->history.size(); ++i)
      rnorms_h[i] = s->history[i];
  PMGX_API_END
}
int pmgx_cg_compute_eigenvalues(pmgx_cg* s, double* eig_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(s && eig_h, "cg_compute_eigenvalues: null argument");
  const int ne = (int)s->alphas.size();
  if (ne < 2)
  {
    pmgx::set_error("Insufficient data to compute eigenvalues"); // src/cg.hpp:125
    return PMGX_ERR_NUMERIC;
  }
  // Lanczos tridiagonal from the CG coefficients (src/cg.hpp:127-135)
  std::vector<double> d(ne, 0.0), e(ne, 0.0);
  for (int i = 0; i < ne; ++i)
    d[i] = 1.0 / s->alphas[i];
  for (int i = 0; i < ne - 1; ++i)
  {
    d[i + 1] += s->betas[i] / s->alphas[i];
    e[i] = std::sqrt(s->betas[i]) / s->alphas[i];
  }
  const int rc = pmgx_tqli(d.data(), e.data(), ne);
  if (rc != PMGX_OK)
    return rc;
  std::sort(d.begin(), d.end());
  for (int i = 0; i < ne; ++i)
    eig_h[i] = d[i];
  PMGX_API_END
}
int pmgx_cg_destroy(pmgx_cg* s)
{
  PMGX_API_BEGIN
  if (s)
  {
    cudaSetDevice(s->ctx->device);
    cudaStreamSynchronize(s->ctx->stream);
    if (s->graph)
      cudaGraphExecDestroy(s->graph);
    if (s->graph_odd)
      cudaGraphExecDestroy(s->graph_odd);
    delete s;
  }
  PMGX_API_END
}

// ---- coarse solver
int pmgx_coarse_create(pmgx_ctx* ctx, pmgx_operator* A, int max_iter, double rtol, pmgx_coarse** out)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(ctx && A && out && max_iter >= 0, "coarse_create: bad arguments");
  std::unique_ptr<pmgx_coarse> cs(new pmgx_coarse());
  cs->ctx = ctx;
  cs->A = A;
  int rc = pmgx_cg_create(ctx, A->n_owned, A->n_ghost, &cs->cg);
  if (rc != PMGX_OK)
    return rc;
  cs->cg->max_iter = max_iter;
  cs->cg->rtol = rtol;
  cs->cg->store = false;
  cs->cg->r.release(); // the coarse variant works in its own slab
  cs->cg->y.release();
  cs->cg->p.release();
  *out = cs.release();
  PMGX_API_END
}
int pmgx_coarse_solve(pmgx_coarse* cs, double* x, const double* b, int* iters_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(cs && x && b, "coarse_solve: null argument");
  PMGX_CUDA(cudaSetDevice(cs->ctx->device));
  const int k = pmgx::cgcg_solve(cs, x, b, false);
  cs->last_iters = k;
  if (iters_h)
    *iters_h = k;
  PMGX_API_END
}
int pmgx_coarse_last_iterations(pmgx_coarse* cs) { return cs ? cs->last_iters : -1; }
int pmgx_coarse_last_status(pmgx_coarse* cs, int* converged_h, double* rel_residual_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(cs, "coarse_last_status: null handle");
  if (converged_h)
    *converged_h = cs->last_converged ? 1 : 0;
  if (rel_residual_h)
    *rel_residual_h = cs->last_rel;
  PMGX_API_END
}

int pmgx_coarse_destroy(pmgx_coarse* cs)
{
  PMGX_API_BEGIN
  if (cs)
  {
    pmgx_cg_destroy(cs->cg);
    delete cs->M;
    delete cs;
  }
  PMGX_API_END
}

// ---- V-cycle
int pmgx_vcycle_create(pmgx_ctx* ctx, int n_levels, pmgx_operator** ops, pmgx_cheb** smoothers,
                       pmgx_interp** interps, const int8_t** bc_markers, pmgx_coarse* coarse, int flags,
                       pmgx_vcycle** out)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(ctx && out && n_levels >= 1 && ops && smoothers && bc_markers, "vcycle_create: bad arguments");
  PMGX_REQUIRE(n_levels == 1 || interps, "vcycle_create: interpolators missing");
  PMGX_CUDA(cudaSetDevice(ctx->device));
  std::unique_ptr<pmgx_vcycle> v(new pmgx_vcycle());
  v->ctx = ctx;
  v->n_levels = n_levels;
  v->flags = flags;
  v->coarse = coarse;
  v->u.resize(n_levels);
  v->r.resize(n_levels);
  v->b.resize(n_levels);
  for (int i = 0; i < n_levels; ++i)
  {
    PMGX_REQUIRE(ops[i] && smoothers[i] && bc_markers[i], "vcycle_create: null level %d", i);
    PMGX_REQUIRE(smoothers[i]->n_owned == ops[i]->n_owned, "Incompatible vector sizes");
    v->ops.push_back(ops[i]);
    v->smoothers.push_back(smoothers[i]);
    v->bc.push_back(bc_markers[i]);
    if (i < n_levels - 1)
    {
      PMGX_REQUIRE(interps[i], "vcycle_create: null interpolator %d", i);
      v->interps.push_back(interps[i]);
    }
    const size_t nt = (size_t)ops[i]->n_owned + ops[i]->n_ghost;
    const bool is_top = i == n_levels - 1 && n_levels > 1;
    for (auto* buf : {&v->u[i], &v->r[i], &v->b[i]})
    {
      if (is_top && buf != &v->r[i])
        continue; // the cycle works on the caller's top-level u and b in place
      buf->alloc(nt);
      if (nt > 0)
        PMGX_CUDA(cudaMemsetAsync(buf->p, 0, nt * sizeof(double), ctx->stream));
    }
  }
  *out = v.release();
  PMGX_API_END
}

int pmgx_vcycle_apply(pmgx_vcycle* v, const double* b_in, double* u_inout, double* rnorm_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(v && b_in && u_inout, "vcycle_apply: null argument");
  pmgx_ctx* c = v->ctx;
  PMGX_CUDA(cudaSetDevice(c->device));
  const int nl = v->n_levels;
  const int top = nl - 1;
  const bool diag = (v->flags & PMGX_VC_DIAGNOSTICS) != 0;
  const bool literal_bc = (v->flags & PMGX_VC_LITERAL_REFERENCE_BC) != 0;
  const bool literal_seq = (v->flags & PMGX_VC_LITERAL_SEQUENCE) != 0;
  v->diagnostics.clear();
  namespace vec = pmgx::vec;
  // The reference copies x into _b[top] and y into _u[top] and back (pmg.hpp:65-68,154); both
  // are full owned+ghost vectors, so the cycle works on the caller's arrays directly.
  std::vector<double*> U(nl);
  std::vector<const double*> B(nl);
  for (int i = 0; i < top; ++i)
    U[i] = v->u[i].p, B[i] = v->b[i].p;
  U[top] = u_inout;
  B[top] = b_in;
  auto residual = [&](int i, bool want_norm) -> double // r = b - A u on level i; optionally its norm
  {
    pmgx_operator* A = v->ops[i];
    A->apply(U[i], v->r[i].p);
    vec::axpy(c, v->r[i].p, -1.0, v->r[i].p, B[i], A->n_owned);
    if (!want_norm)
      return 0.0;
    return std::sqrt(vec::dot(c, v->r[i].p, v->r[i].p, A->n_owned));
  };
  for (int i = 0; i < top; ++i) // pmg.hpp:63-64
    vec::set(c, U[i], (long long)v->ops[i]->n_owned + v->ops[i]->n_ghost, 0.0);

  for (int i = top; i > 0; --i)
  {
    if (diag)
      v->diagnostics.push_back(residual(i, true));                                // :76-80
    // below the top level u is zero on the way down: the smoother's first apply is skipped.
    // The smoother's recurrence already holds r = b - A u of its final iterate
    // (src/chebyshev.hpp:73-77; the reference recomputes it with one more apply, :86-89), and
    // the last r -= q is folded into the restriction's gather.
    const pmgx::ChebResidual want = literal_seq ? pmgx::CHEB_R_FULL : (diag ? pmgx::CHEB_R_FULL : pmgx::CHEB_R_SPLIT);
    pmgx::cheb_solve(v->smoothers[i], v->ops[i], U[i], B[i], nullptr, !literal_seq && i < top, want); // :83
    double* rfine = v->r[i].p;
    const double* rsub = nullptr;
    if (literal_seq)
    {
      const double rn = residual(i, diag);                                        // :86-89
      if (diag)
        v->diagnostics.push_back(rn);
    }
    else
    {
      rfine = v->smoothers[i]->r.p;
      if (want == pmgx::CHEB_R_SPLIT && v->smoothers[i]->max_iter > 0)
        rsub = v->smoothers[i]->q.p;
      if (diag)
        v->diagnostics.push_back(std::sqrt(vec::dot(c, rfine, rfine, v->ops[i]->n_owned)));
    }
    pmgx::interp_restrict(v->interps[i - 1], rfine, rsub, v->b[i - 1].p);          // :92
    if (!literal_bc && i - 1 > 0) // quirk Q9: keep Dirichlet rows of intermediate levels clean
      vec::mask_bc(c, v->b[i - 1].p, v->bc[i - 1], v->ops[i - 1]->n_owned);
  }
  if (nl > 1)
    vec::mask_bc(c, v->b[0].p, v->bc[0], v->ops[0]->n_owned);                      // :100-103
  else
  {
    // single level: the reference masks its private copy of b; keep the caller's b intact
    vec::copy(c, v->b[0].p, b_in, v->ops[0]->n_owned);
    vec::mask_bc(c, v->b[0].p, v->bc[0], v->ops[0]->n_owned);
    B[0] = v->b[0].p;
  }
  const pmgx::ChebResidual post = literal_seq ? pmgx::CHEB_R_FULL : pmgx::CHEB_R_NONE;
  if (v->coarse && nl > 1)
  {
    v->coarse->last_iters = pmgx::cgcg_solve(v->coarse, U[0], B[0], true); // :106-107 (u[0] = 0)
  }
  else
    pmgx::cheb_solve(v->smoothers[0], v->ops[0], U[0], B[0], nullptr, !literal_seq && nl > 1, post); // :109
  if (diag)
    v->diagnostics.push_back(residual(0, true));                                  // :114-117

  for (int i = 0; i < top; ++i)
  {
    // u[i+1] += P u[i]: the reference prolongs into du and adds (:123-129); the sum is formed in
    // the prolongation's store
    pmgx::interp_prolong(v->interps[i], U[i], U[i + 1], true);
    if (diag)
      v->diagnostics.push_back(residual(i + 1, true));                            // :132-135
    pmgx::cheb_solve(v->smoothers[i + 1], v->ops[i + 1], U[i + 1], B[i + 1], nullptr, false, post); // :138
    if (diag && i + 1 < top)
      v->diagnostics.push_back(residual(i + 1, true));                            // :141-144
  }
  if (rnorm_h || diag)
  {
    const double rn = residual(top, true);                                        // :141-149
    if (rnorm_h)
      *rnorm_h = rn;
    if (diag)
      v->diagnostics.push_back(rn);
  }
  PMGX_API_END
}

int pmgx_vcycle_get_diagnostics(pmgx_vcycle* v, double* out_h, int cap, int* n_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(v, "vcycle_get_diagnostics: null handle");
  const int n = (int)v->diagnostics.size();
  if (n_h)
    *n_h = n;
  if (out_h)
    for (int i = 0; i < n && i < cap; ++i)
      out_h[i] = v->diagnostics[i];
  PMGX_API_END
}

int pmgx_vcycle_destroy(pmgx_vcycle* v)
{
  PMGX_API_BEGIN
  if (v)
  {
    cudaSetDevice(v->ctx->device);
    cudaStreamSynchronize(v->ctx->stream);
    delete v;
  }
  PMGX_API_END
}
}
