// Solver state behind the opaque C handles, shared between solvers.cu (Chebyshev, CG, V-cycle) and
// amg.cu (the multilevel coarse solver, which smooths with the same Chebyshev code and is the
// preconditioner of the coarse PCG).
#pragma once
#include "common.hpp"
#include "operator.hpp"

// acc::Chebyshev state (src/chebyshev.hpp:94-105)
struct pmgx_cheb
{
  pmgx_ctx* ctx = nullptr;
  int n_owned = 0, n_ghost = 0;
  double eig_min = 0.0, eig_max = 1.0;
  int max_iter = 0;
  pmgx::DevBuf<double> z, q, r; // work vectors (owned + ghost), src/chebyshev.hpp:101-105
  pmgx::DevBuf<double> z2;      // second z buffer of the fused (row-complete operator) path, allocated on first use
};

namespace pmgx
{
// what the caller of cheb_solve needs of the recurrence residual r = b - A x_final afterwards:
//   CHEB_R_NONE   nothing: the last iteration of the reference (one apply + one pass that only
//                 feed r and a z nobody reads, chebyshev.hpp:76-83) is dropped; x is bit-identical
//   CHEB_R_FULL   s->r holds r
//   CHEB_R_SPLIT  s->r - s->q is r (the caller folds the subtraction into its own gather)
enum ChebResidual
{
  CHEB_R_NONE = 0,
  CHEB_R_FULL = 1,
  CHEB_R_SPLIT = 2
};
// x <- Chebyshev(A, x, b). hist: max_iter+1 residual norms or nullptr.
void cheb_solve(pmgx_cheb* s, pmgx_operator* A, double* x, const double* b, double* hist, bool x_is_zero = false,
                ChebResidual final_r = CHEB_R_FULL);

// u = M^-1 r for the coarse PCG; r and u are owned+ghost vectors of the solver's level
struct Precond
{
  virtual ~Precond() {}
  virtual void apply(const double* r, double* u) = 0;
};
} // namespace pmgx

// acc::CGSolver state (src/cg.hpp:225-248) + the single-reduction coarse variant's slab and graph
struct pmgx_cg
{
  pmgx_ctx* ctx = nullptr;
  int n_owned = 0, n_ghost = 0;
  int max_iter = 0;
  double rtol = 0.0;
  bool store = false;
  pmgx_vcycle* precond = nullptr; // borrowed; null: Jacobi (diag^-1 of the operator, src/cg.hpp:154)
  pmgx::DevBuf<double> r, y, p; // src/cg.hpp:241-244
  pmgx::DevBuf<double> slab;    // r, w, p, u, s of the single-reduction coarse variant, contiguous (lazy)
  // CUDA graph of one block of `graph_len` coarse iterations (captured from the stream on first use,
  // replayed between the host's convergence checks): the ~8 small launches and 4 cross-stream
  // events of an iteration cost more in launch gaps than the kernels of a 1.6 M-dof level run
  cudaGraphExec_t graph = nullptr, graph_odd = nullptr; // blocks starting at an even / odd iteration
  const void* graph_key[3] = {nullptr, nullptr, nullptr}; // operator, x, block length
  int graph_launches = 0;
  bool graph_off = false;
  std::vector<double> alphas, betas, residuals; // stored coefficients (:213-218)
  std::vector<double> history;                  // every iteration's r.M^-1 r
  double rnorm0 = 0.0;
};

// CoarseSolverType (src/amg.hpp:9-119): PCG on the assembled operator; M = Jacobi or the AMG cycle
struct pmgx_coarse
{
  pmgx_ctx* ctx = nullptr;
  pmgx_operator* A = nullptr;
  pmgx_cg* cg = nullptr;
  pmgx::Precond* M = nullptr; // owned; null: Jacobi
  int check_every = 8;        // host looks at r.M^-1 r every this many iterations
  int last_iters = 0;
  bool last_converged = false;
  double last_rel = 0.0;      // sqrt(r.M^-1 r / r0.M^-1 r0) at the last check
};

namespace pmgx
{
int cgcg_solve(pmgx_coarse* cs, double* x, const double* b, bool x_is_zero);
// rectangular CSR product y = M x, 32 lanes per row, for long rows (the AMG restriction; csr.cu)
void spmv_rect(pmgx_ctx* c, int n_rows, const int32_t* row_ptr, const int32_t* cols, const double* vals,
               const double* x, double* y);
// y += M x for a matrix stored as sliced ELL (32-row slices, column-major inside a slice; padding: value 0,
// column 0): thread per row, for short rows (the AMG prolongator)
void spmv_sell_rect(pmgx_ctx* c, int n_rows, const long long* slice_ptr, const int32_t* cols, const double* vals,
                    const double* x, double* y);
} // namespace pmgx
