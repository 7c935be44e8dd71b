// C++ host driver of the p-multigrid Poisson solve, written against the reference's class
// names through include/pmgx/dolfinx_acc_compat.hpp.  Mirrors examples/pmg/main.cpp of the
// reference (solve_problem, :44-384): box mesh sized by the fit routine (:412-435), one space
// per degree, matrix-free operators with Dirichlet marker, lambda_max from a 20-iteration CG
// with b = 1 (:306-330), Chebyshev(2) smoothers, element-local interpolators, P1 CSR coarse
// solver behind CoarseSolverType, then `niter` V-cycles with the residual printed (:359-367).
// Only the DOLFINx set-up (mesh, function spaces, assembly of b) is swapped for the box-mesh
// helpers of the C ABI.
//
//   pmg_main [--ndofs N] [--degrees 1,2,4] [--niter 10] [--perturb 0.0] [--coarse-its 60] [--batch_size 0]
// --batch_size N > 0: every MatFreeLaplacian keeps no geometry and recomputes it in each apply (the
// reference's option of the same name; N itself only selects the mode).
// Multi-GPU: one process per GPU with RANK / WORLD_SIZE / LOCAL_RANK in the environment and
// --idfile PATH on a shared filesystem (rank 0 writes the NCCL id there; the reference uses
// MPI for this, which this image does not have).
#include "box_setup.hpp"

using T = double;
using namespace dolfinx;
using DeviceVector = acc::Vector<T, acc::Device::CUDA>;
using box::Space;

int main(int argc, char** argv)
{
  long long ndofs = 50000; // per rank, like the reference's default (:405)
  std::vector<int> degrees = {1, 2, 4};
  int niter = 10, coarse_its = 60;
  std::size_t batch_size = 0;
  double perturb = 0.0, coarse_rtol = 1e-5; // PETSc default rtol of the reference's coarse KSP (src/amg.hpp:40)
  std::string idfile;
  for (int i = 1; i < argc; ++i)
  {
    auto next = [&]() -> const char*
    {
      if (i + 1 >= argc)
        throw std::runtime_error(std::string("missing value for ") + argv[i]);
      return argv[++i];
    };
    if (!std::strcmp(argv[i], "--ndofs"))
      ndofs = (long long)std::atof(next());
    else if (!std::strcmp(argv[i], "--niter"))
      niter = std::atoi(next());
    else if (!std::strcmp(argv[i], "--perturb"))
      perturb = std::atof(next());
    else if (!std::strcmp(argv[i], "--coarse-its"))
      coarse_its = std::atoi(next());
    else if (!std::strcmp(argv[i], "--idfile"))
      idfile = next();
    else if (!std::strcmp(argv[i], "--batch_size"))
      batch_size = (std::size_t)std::atoll(next());
    else if (!std::strcmp(argv[i], "--degrees"))
    {
      degrees.clear();
      std::stringstream ss(next());
      for (std::string tok; std::getline(ss, tok, ',');)
        degrees.push_back(std::atoi(tok.c_str()));
    }
    else
    {
      std::printf("usage: %s [--ndofs N] [--degrees 1,2,4] [--niter 10] [--perturb p] [--coarse-its k] "
                  "[--batch_size N] [--idfile path]\n", argv[0]);
      return std::strcmp(argv[i], "--help") ? 1 : 0;
    }
  }
  try
  {
    const int rank = box::env_int("RANK", 0), nranks = box::env_int("WORLD_SIZE", 1);
    const int local = box::env_int("LOCAL_RANK", 0);
    std::vector<char> id;
    box::exchange_nccl_id(rank, nranks, idfile, id);
    auto ctx = std::make_shared<pmgx::Context>(local, rank, nranks, nranks > 1 ? id.data() : nullptr);

    // ---- mesh (examples/pmg/main.cpp:412-451, src/mesh.hpp:16-143)
    box::Mesh mesh(ndofs, degrees.back(), rank, nranks, perturb, 2.0 /* kappa, :79 */);
    const std::vector<int>& lcells = mesh.lcells;
    const std::vector<int>& bcells = mesh.bcells;
    if (rank == 0)
      std::printf("mesh %d x %d x %d cells, %d rank(s), cells/rank %d (lcells %zu, bcells %zu)\n", mesh.nxyz[0],
                  mesh.nxyz[1], mesh.nxyz[2], nranks, mesh.n_cells, lcells.size(), bcells.size());

    // ---- spaces, maps, device dofmaps and BC markers (:83-124,199-256)
    std::vector<Space> V(degrees.size());
    std::vector<std::shared_ptr<const pmgx::IndexMap>> maps;
    for (size_t i = 0; i < degrees.size(); ++i)
    {
      mesh.make_space(ctx, degrees[i], V[i]);
      maps.push_back(V[i].map);
      if (rank == 0)
        std::printf("level %zu: P%d, %lld dofs (rank 0: %d owned + %d ghost)\n", i, V[i].degree, V[i].n_global,
                    V[i].map->size_local(), V[i].map->num_ghosts());
    }

    // ---- operators (:258-287); the matrix-free diagonal replaces the per-level CSR assembly (:274-279)
    using FineOperator = acc::MatFreeLaplacian<T>;
    std::vector<std::shared_ptr<FineOperator>> operators;
    for (Space& s : V)
      operators.push_back(std::make_shared<FineOperator>(s.degree, mesh.kappa.span(), s.dofmap.span(), mesh.xgeom.span(),
                                                         mesh.geometry_dofmap.span(), std::span<const T>(),
                                                         std::span<const T>(), lcells, bcells, s.bc.span(),
                                                         batch_size));

    // ---- right-hand side on the finest level (:289-300, examples/pmg/poisson.py:6-8,30)
    Space& top = V.back();
    const int nt = top.map->size_local() + top.map->num_ghosts();
    std::vector<double> f((size_t)nt);
    const double kx = 2, ky = 3, kz = 4, kap = 2.0, pi = M_PI;
    for (int i = 0; i < nt; ++i)
      f[i] = kap * pi * pi * (kx * kx + ky * ky + kz * kz) * std::sin(kx * pi * top.coords[3 * i])
             * std::sin(ky * pi * top.coords[3 * i + 1]) * std::sin(kz * pi * top.coords[3 * i + 2]);
    pmgx::DeviceArray<double> fvals(f);
    DeviceVector b(maps.back(), 1);
    pmgx::check(pmgx_laplacian_rhs(operators.back()->handle(maps.back()), fvals.p, 0.0, b.mutable_array().data()));
    if (rank == 0)
      std::printf("b.norm = %.12e\n", acc::norm(b));
    else
      acc::norm(b);

    // ---- Chebyshev smoothers from CG eigenvalue estimates (:306-330)
    std::vector<std::shared_ptr<acc::Chebyshev<DeviceVector>>> smoothers(V.size());
    for (size_t i = 0; i < V.size(); ++i)
    {
      acc::CGSolver<DeviceVector> cg(maps[i], 1);
      cg.set_max_iterations(20);
      cg.set_tolerance(1e-6);
      cg.store_coefficients(true);
      DeviceVector x(maps[i], 1), y(maps[i], 1);
      x.set(T{0.0});
      y.set(T{1.0});
      [[maybe_unused]] int its = cg.solve(*operators[i], x, y, false);
      std::vector<T> eign = cg.compute_eigenvalues();
      if (rank == 0)
        std::printf("Eigenvalues level %zu: %.10f - %.10f (CG its %d)\n", i, eign.front(), eign.back(), its);
      std::array<T, 2> eig_range = {0.1 * eign.back(), 1.1 * eign.back()};
      smoothers[i] = std::make_shared<acc::Chebyshev<DeviceVector>>(maps[i], 1, eig_range);
      smoothers[i]->set_max_iterations(2);
    }

    // ---- interpolators (:336-343)
    std::vector<std::shared_ptr<Interpolator<T>>> interpolators(V.size() - 1);
    std::vector<std::int32_t> lc32(lcells.begin(), lcells.end()), bc32(bcells.begin(), bcells.end());
    for (size_t i = 0; i + 1 < V.size(); ++i)
      interpolators[i] = std::make_shared<Interpolator<T>>(pmgx::Element(V[i].degree), pmgx::Element(V[i + 1].degree),
                                                           V[i].dofmap.span(), V[i + 1].dofmap.span(), lc32, bc32);

    // ---- coarse solver on the assembled P1 matrix (:128-130; src/amg.hpp)
    auto A0 = std::make_shared<acc::MatrixOperator<T>>(*operators[0], maps[0]);
    auto coarse_solver = std::make_shared<CoarseSolverType<T>>(A0, maps[0], coarse_its, coarse_rtol);
    if (rank == 0)
      std::printf("coarse matrix: %zu non-zeros on rank 0\n", A0->nnz());

    // ---- PMG (:345-356)
    using SolverType = acc::Chebyshev<DeviceVector>;
    using PMG = acc::MultigridPreconditioner<DeviceVector, FineOperator, SolverType, CoarseSolverType<T>, Interpolator<T>>;
    PMG pmg(maps, 1, V[0].bc.span());
    std::vector<std::span<const std::int8_t>> markers;
    for (Space& s : V)
      markers.push_back(s.bc.span());
    pmg.set_bc_markers(markers);
    pmg.set_solvers(smoothers);
    pmg.set_operators(operators);
    pmg.set_coarse_solver(coarse_solver);
    pmg.set_interpolators(interpolators);

    DeviceVector x(maps.back(), 1);
    x.set(T{0.0});
    const double bnorm = acc::norm(b);
    ctx->synchronize();
    const auto t0 = std::chrono::steady_clock::now();
    double rnorm = 0;
    for (int i = 0; i < niter; ++i) // :362-367
    {
      pmg.apply(b, x, true);
      rnorm = pmg.last_residual_norm();
      if (rank == 0)
        std::printf("PMG iteration %2d: rnorm after PMG = %.6e (relative %.3e)\n", i + 1, rnorm, rnorm / bnorm);
    }
    ctx->synchronize();
    const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (rank == 0)
      std::printf("%d V-cycles (incl. residual norms) in %.3f s; %lld fine dofs; final relative residual %.3e\n", niter,
                  dt, top.n_global, rnorm / bnorm);
    return rnorm / bnorm < 1.0 ? 0 : 2;
  }
  catch (const std::exception& e)
  {
    std::fprintf(stderr, "pmg_main: %s\n", e.what());
    return 1;
  }
}
