// Device cycle of the smoothed-aggregation coarse solver: the preconditioner of the coarse PCG behind
// CoarseSolverType::solve, where the reference runs PETSc KSPCG + BoomerAMG (src/amg.hpp:33-47,67-113).
//
// The hierarchy comes from amg_setup.cpp (host, collective).  Everything the cycle runs already exists
// in this library: the CSR SpMV with its owned/ghost column split and overlapped halo (csr.cu), the
// 4th-kind Chebyshev/Jacobi smoother with its dead-iteration elimination (solvers.cu), the
// peer-memory halo (halo.cu).  Prolongation and restriction are rectangular CSR products (P and the owned
// rows of P^T, stored explicitly: a gather, so the restriction is deterministic) behind one forward halo
// update each, because the smoothed prolongator reaches across partition interfaces; the coarsest level
// is gathered with an all-to-all halo plan and multiplied by this rank's rows of the dense inverse.
// One V(nu,nu) cycle: per level 2 nu SpMVs + 2 transfers, no host synchronisation anywhere, so the
// coarse PCG captures whole iterations into a CUDA graph (solvers.cu, cgcg_solve).
#include "common.hpp"
#include "operator.hpp"
#include "csr.hpp"
#include "solvers.hpp"
#include "amg.hpp"

#include <algorithm>
#include <cstdlib>
#include <cstring>

namespace pmgx
{
namespace
{
// x[row] = sum_c inv[row][c] * b[c]; one warp per row, b = [owned | gathered] (n_cols entries)
__global__ void __launch_bounds__(256)
k_dense_rows(int n_rows, int n_cols, const double* __restrict__ inv, const double* __restrict__ b,
             double* __restrict__ x)
{
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= n_rows)
    return;
  const double* r = inv + (size_t)row * n_cols;
  double s = 0.0;
  for (int c = lane; c < n_cols; c += 32)
    s = fma(r[c], b[c], s);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
    s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0)
    x[row] = s;
}

// out[g] = in[perm[g]]
__global__ void k_permute(int n, const int32_t* __restrict__ perm, const double* __restrict__ in, double* __restrict__ out)
{
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < n)
    out[g] = in[perm[g]];
}

// short-row rectangular matrix as sliced ELL (thread per row): the prolongator has 1..8 entries per row, with
// 4 lanes per CSR row its apply is a chain of dependent loads per row (85 us at 1.59 M rows under ncu, as much
// as a level-0 SpMV that moves six times the bytes)
struct RectSell
{
  int n_rows = 0;
  DevBuf<long long> slice_ptr;
  DevBuf<int32_t> cols;
  DevBuf<double> vals;
  void upload(const amg::Csr& M, cudaStream_t st)
  {
    n_rows = M.n_rows;
    const int ns = (n_rows + 31) / 32;
    std::vector<long long> sp((size_t)ns + 1, 0);
    for (int s = 0; s < ns; ++s)
    {
      int w = 0;
      for (int r = s * 32; r < std::min(n_rows, s * 32 + 32); ++r)
        w = std::max(w, (int)(M.ptr[r + 1] - M.ptr[r]));
      sp[s + 1] = sp[s] + (long long)w * 32;
    }
    std::vector<int32_t> c((size_t)std::max<long long>(sp[ns], 1), 0);
    std::vector<double> v((size_t)std::max<long long>(sp[ns], 1), 0.0);
    for (int r = 0; r < n_rows; ++r)
      for (int32_t j = M.ptr[r], k = 0; j < M.ptr[r + 1]; ++j, ++k)
      {
        const size_t p = (size_t)sp[r >> 5] + (size_t)k * 32 + (r & 31);
        c[p] = M.cols[j];
        v[p] = M.vals[j];
      }
    slice_ptr.upload(sp.data(), sp.size(), st);
    cols.upload(c.data(), c.size(), st);
    vals.upload(v.data(), v.size(), st);
  }
};

struct RectCsr
{
  int n_rows = 0;
  DevBuf<int32_t> ptr, cols;
  DevBuf<double> vals;
  void upload(const amg::Csr& M, cudaStream_t st)
  {
    n_rows = M.n_rows;
    ptr.upload(M.ptr.data(), M.ptr.size(), st);
    cols.upload(M.cols.data(), M.cols.size(), st);
    vals.upload(M.vals.data(), M.vals.size(), st);
  }
};

pmgx_halo* make_halo(pmgx_ctx* c, int n_owned, int n_ghost, const amg::Plan& p)
{
  if (c->nranks == 1)
    return nullptr;
  pmgx_halo* h = nullptr;
  const int rc = pmgx_halo_create(c, n_owned, n_ghost, (int)p.send_ranks.size(), p.send_ranks.data(), p.send_offsets.data(),
                                  p.send_idx.data(), (int)p.recv_ranks.size(), p.recv_ranks.data(), p.recv_offsets.data(),
                                  p.recv_idx.data(), &h);
  if (rc != PMGX_OK)
    throw Error{rc};
  // latency-bound exchanges: stay on the compute stream (PMGX_AMG_SINGLE_STREAM=0: dual-stream like level 0)
  static const bool ss = !(getenv("PMGX_AMG_SINGLE_STREAM") && atoi(getenv("PMGX_AMG_SINGLE_STREAM")) == 0);
  h->single_stream = ss && h->p2p && h->n_send() + h->n_recv() <= 65536;
  return h;
}

struct AmgPrecond : Precond
{
  struct Lv
  {
    int n_owned = 0, n_ghost = 0;
    long long nnz = 0;
    pmgx_operator* A = nullptr;
    bool own_A = false;
    pmgx_operator* A_lp = nullptr; // owned: reduced-storage twin used by the smoother (level 0 only)
    pmgx_halo* halo = nullptr; // owned (levels >= 1)
    pmgx_halo* halo_v = nullptr; // borrowed: forward-scatter plan of this level's vectors (level 0: the operator's)
    pmgx_cheb* sm = nullptr;
    RectCsr R;                 // from this level to the next coarser one (rows of P^T: long rows, 32 lanes per row)
    RectSell P;                // back (short rows, thread per row)
    DevBuf<double> x, b;       // levels >= 1 (and the private b of a dense level)
    DevBuf<double> x2, r2;     // second coarse visit of a W-cycle (levels >= 1)
    long long nnz_p = 0;
    bool dense = false;
    int n_global = 0;
    DevBuf<double> inv;
    pmgx_halo* gather = nullptr; // owned
    // first replicated level: all-gather of the restricted residual, then the canonical ordering
    bool repl_first = false;
    int n_mine = 0;
    pmgx_halo* repl_gather = nullptr; // owned
    DevBuf<double> bg;                // [mine | the others in rank order]
    DevBuf<int32_t> perm;             // canonical index -> position in bg
  };
  pmgx_ctx* ctx = nullptr;
  std::vector<Lv> lv;
  int nu = 2;
  int gamma = 1; // cycle index: 1 = V, 2 = W (two coarse visits; the small levels are latency, not bandwidth)
  int gamma_from = 0; // first level whose coarse level is visited gamma times

  ~AmgPrecond() override
  {
    for (Lv& L : lv)
    {
      if (L.sm)
        pmgx_cheb_destroy(L.sm);
      if (L.A_lp)
        pmgx_operator_destroy(L.A_lp);
      if (L.own_A && L.A)
        pmgx_operator_destroy(L.A);
      if (L.halo)
        pmgx_halo_destroy(L.halo);
      if (L.gather)
        pmgx_halo_destroy(L.gather);
      if (L.repl_gather)
        pmgx_halo_destroy(L.repl_gather);
    }
  }

  void cycle(int l, const double* b, double* x)
  {
    Lv& L = lv[l];
    if (l + 1 == (int)lv.size())
    {
      if (L.dense)
      {
        double* bb = L.b.p; // private: its ghost block receives the other ranks' entries
        if (b != bb)
          vec::copy(ctx, bb, b, L.n_owned);
        if (L.gather)
        {
          halo_fwd_begin(L.gather, bb);
          halo_fwd_end(L.gather, bb);
        }
        if (L.n_owned > 0)
        {
          k_dense_rows<<<(L.n_owned * 32 + 255) / 256, 256, 0, ctx->stream>>>(L.n_owned, L.n_global, L.inv.p, bb, x);
          check_launch("k_dense_rows");
          count_launch(ctx);
        }
      }
      else // no dense inverse (level too large): smooth instead
        cheb_solve(L.sm, L.A, x, b, nullptr, true, CHEB_R_NONE);
      return;
    }
    Lv& C = lv[l + 1];
    pmgx_operator* As = L.A_lp ? L.A_lp : L.A;
    cheb_solve(L.sm, As, x, b, nullptr, true, CHEB_R_FULL);           // pre-smoothing from x = 0; sm->r = b - A x
    if (L.halo_v) // the rows of P^T this rank owns reach into the neighbours' fine dofs
    {
      halo_fwd_begin(L.halo_v, L.sm->r.p);
      halo_fwd_end(L.halo_v, L.sm->r.p);
    }
    if (C.repl_first)
    {
      // the next level lives completely on every rank: my part of b_c, all-gather, canonical order
      spmv_rect(ctx, C.n_mine, L.R.ptr.p, L.R.cols.p, L.R.vals.p, L.sm->r.p, C.bg.p, false, 32);
      halo_fwd_begin(C.repl_gather, C.bg.p);
      halo_fwd_end(C.repl_gather, C.bg.p);
      k_permute<<<(C.n_owned + 255) / 256, 256, 0, ctx->stream>>>(C.n_owned, C.perm.p, C.bg.p, C.b.p);
      check_launch("k_permute");
      count_launch(ctx);
    }
    else
      spmv_rect(ctx, C.n_owned, L.R.ptr.p, L.R.cols.p, L.R.vals.p, L.sm->r.p, C.b.p, false, 32); // b_c = P^T r
    cycle(l + 1, C.b.p, C.x.p);
    if (gamma == 2 && l >= gamma_from && l + 2 < (int)lv.size())
    {
      // W-cycle: a second visit on the coarse residual, x_c += B_c (b_c - A_c x_c)  (symmetric: 2B - BAB)
      C.A->apply(C.x.p, C.r2.p);
      vec::axpy(ctx, C.r2.p, -1.0, C.r2.p, C.b.p, C.n_owned);
      cycle(l + 1, C.r2.p, C.x2.p);
      vec::axpy(ctx, C.x.p, 1.0, C.x2.p, C.x.p, C.n_owned);
    }
    if (C.halo_v) // ... and P interpolates from the neighbours' aggregates
    {
      halo_fwd_begin(C.halo_v, C.x.p);
      halo_fwd_end(C.halo_v, C.x.p);
    }
    spmv_sell_rect(ctx, L.n_owned, L.P.slice_ptr.p, L.P.cols.p, L.P.vals.p, C.x.p, x, true); // x += P x_c
    cheb_solve(L.sm, As, x, b, nullptr, false, CHEB_R_NONE);          // post-smoothing (same polynomial: M is symmetric)
  }

  void apply(const double* r, double* u) override { cycle(0, r, u); }
};

// forward-scatter plan of an existing halo, back on the host
amg::Plan plan_of(pmgx_halo* h)
{
  amg::Plan p;
  if (!h)
    return p;
  p.send_ranks = h->send_ranks;
  p.send_offsets = h->send_offsets;
  p.recv_ranks = h->recv_ranks;
  p.recv_offsets = h->recv_offsets;
  if (p.send_offsets.empty())
    p.send_offsets.assign(1, 0);
  if (p.recv_offsets.empty())
    p.recv_offsets.assign(1, 0);
  p.send_idx.resize((size_t)h->n_send());
  p.recv_idx.resize((size_t)h->n_recv());
  if (!p.send_idx.empty())
    PMGX_CUDA(cudaMemcpy(p.send_idx.data(), h->send_idx.p, p.send_idx.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
  if (!p.recv_idx.empty())
    PMGX_CUDA(cudaMemcpy(p.recv_idx.data(), h->recv_idx.p, p.recv_idx.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
  return p;
}
} // namespace
} // namespace pmgx

using pmgx::AmgPrecond;

extern "C"
{
int pmgx_coarse_create_amg(pmgx_ctx* ctx, pmgx_operator* A, int max_iter, double rtol, int nu, int min_coarse,
                           int max_levels, pmgx_coarse** out)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(ctx && A && out && max_iter >= 0, "coarse_create_amg: bad arguments");
  PMGX_REQUIRE(A->kind == pmgx_operator::CSR, "coarse_create_amg: the operator must be an assembled CSR operator");
  PMGX_REQUIRE(nu >= 1 && nu <= 8, "coarse_create_amg: nu must be in 1..8");
  PMGX_CUDA(cudaSetDevice(ctx->device));
  if (min_coarse <= 0)
    min_coarse = 600;
  if (max_levels <= 0)
    max_levels = 12;
  auto* Ac = static_cast<pmgx::CsrOperator*>(A);
  PMGX_REQUIRE(ctx->nranks == 1 || Ac->halo || Ac->n_ghost == 0, "coarse_create_amg: the operator has ghosts but no halo");
  // level-0 matrix and its halo plan, back on the host; rows sorted by column for the set-up
  pmgx::amg::Csr A0;
  A0.ptr.resize((size_t)Ac->n_owned + 1);
  A0.cols.resize((size_t)Ac->nnz);
  A0.vals.resize((size_t)Ac->nnz);
  {
    const int rc = pmgx_csr_get(A, A0.ptr.data(), A0.cols.data(), A0.vals.data());
    if (rc != PMGX_OK)
      return rc;
    std::vector<std::pair<int32_t, double>> row;
    for (int i = 0; i < Ac->n_owned; ++i)
    {
      bool sorted = true;
      for (int32_t j = A0.ptr[i] + 1; j < A0.ptr[i + 1] && sorted; ++j)
        sorted = A0.cols[j - 1] < A0.cols[j];
      if (sorted)
        continue;
      row.clear();
      for (int32_t j = A0.ptr[i]; j < A0.ptr[i + 1]; ++j)
        row.emplace_back(A0.cols[j], A0.vals[j]);
      std::sort(row.begin(), row.end());
      for (size_t t = 0; t < row.size(); ++t)
        A0.cols[A0.ptr[i] + t] = row[t].first, A0.vals[A0.ptr[i] + t] = row[t].second;
    }
  }
  // Stored zeros: the device assembly keeps the full pattern of the element matrices (27 entries per row at P1),
  // of which 7 (affine boxes, collocated quadrature) to 19 are non-zero.  The set-up below gets the pattern (its
  // aggregates follow it: 3 x 3 x 3 blocks); the SpMVs of the solve -- PCG and the level-0 smoother, the only ones
  // that stream from HBM -- run on a copy without the zeros: the same sums minus exact-zero products.
  pmgx::amg::Csr Az;
  if (Ac->n_owned > 0)
  {
    A0.n_rows = Ac->n_owned;
    A0.n_cols = Ac->n_owned + Ac->n_ghost;
    Az = pmgx::amg::drop_stored_zeros(A0);
    if (Az.nnz() * 5 > A0.nnz() * 4) // less than a fifth to gain: not worth a second copy
      Az = pmgx::amg::Csr();
  }
  const pmgx::amg::Plan plan0 = pmgx::plan_of(Ac->halo);
  pmgx::amg::Comm cm;
  cm.rank = ctx->rank;
  cm.nranks = ctx->nranks;
  cm.allgather = [ctx](const void* mine, size_t bytes, void* all)
  {
    std::vector<char> buf;
    pmgx::p2p::allgather_bytes(ctx, mine, bytes, buf);
    std::memcpy(all, buf.data(), bytes * (size_t)ctx->nranks);
  };
  pmgx::amg::Hierarchy H;
  pmgx::amg::setup(H, std::move(A0), Ac->n_owned, Ac->n_ghost, plan0, cm, min_coarse, max_levels);

  std::unique_ptr<AmgPrecond> M(new AmgPrecond());
  M->ctx = ctx;
  M->nu = nu;
  // A/B switches (defaults are the measured winners, DESIGN.md section 3.3)
  int nu_coarse = nu;
  if (const char* e = getenv("PMGX_AMG_NU_COARSE"))
    nu_coarse = std::min(std::max(atoi(e), 1), 8);
  if (const char* e = getenv("PMGX_AMG_GAMMA"))
    M->gamma = atoi(e) == 2 ? 2 : 1;
  if (const char* e = getenv("PMGX_AMG_GAMMA_FROM"))
    M->gamma_from = std::max(atoi(e), 0);
  const bool use_lp = !(getenv("PMGX_AMG_LP") && atoi(getenv("PMGX_AMG_LP")) == 0);
  // first level whose smoother runs the fused SpMV + Chebyshev kernels: every level.  Level 0's smoother runs
  // the thread-per-row sliced-ELL twin, whose epilogue needs no barrier (DESIGN.md section 3.3)
  const int fuse_from = getenv("PMGX_AMG_FUSE_FROM") ? atoi(getenv("PMGX_AMG_FUSE_FROM")) : 0;
  const int nl = (int)H.levels.size();
  M->lv.resize((size_t)nl);
  for (int l = 0; l < nl; ++l)
  {
    pmgx::amg::Level& L = H.levels[l];
    AmgPrecond::Lv& D = M->lv[l];
    D.n_owned = L.n_owned;
    D.n_ghost = L.n_ghost;
    D.nnz = L.A.nnz();
    const bool last = l + 1 == nl;
    if (l == 0)
    {
      D.A = A; // the caller's operator and halo
      D.halo_v = Ac->halo;
      if (!Az.ptr.empty())
      { // ... or its copy without the stored zeros (same halo, same vectors)
        std::vector<int32_t> off((size_t)Ac->n_owned);
        for (int i = 0; i < Ac->n_owned; ++i)
        {
          int32_t j = Az.ptr[i];
          while (j < Az.ptr[i + 1] && Az.cols[j] < Ac->n_owned)
            ++j;
          off[i] = j;
        }
        pmgx_operator* Acmp = nullptr;
        const int rc = pmgx_csr_create(ctx, Ac->n_owned, Ac->n_ghost, Az.ptr.data(), off.data(), Az.cols.data(),
                                       Az.vals.data(), Ac->halo, &Acmp);
        if (rc != PMGX_OK)
          return rc;
        D.A = Acmp;
        D.own_A = true;
      }
    }
    else
    {
      if (!L.replicated)
      {
        D.halo = pmgx::make_halo(ctx, L.n_owned, L.n_ghost, L.plan); // collective: same order on every rank
        D.halo_v = D.halo;
      }
      else if (L.n_mine > 0 || !L.gather_perm.empty())
      {
        // first replicated level (collective as well)
        D.repl_first = true;
        D.n_mine = L.n_mine;
        D.repl_gather = pmgx::make_halo(ctx, L.n_mine, L.n_owned - L.n_mine, L.repl_plan);
        D.bg.alloc((size_t)std::max(L.n_owned, 1));
        PMGX_CUDA(cudaMemsetAsync(D.bg.p, 0, (size_t)std::max(L.n_owned, 1) * sizeof(double), ctx->stream));
        D.perm.upload(L.gather_perm.data(), L.gather_perm.size(), ctx->stream);
      }
      std::vector<int32_t> off((size_t)L.n_owned);
      for (int i = 0; i < L.n_owned; ++i)
      {
        int32_t j = L.A.ptr[i];
        while (j < L.A.ptr[i + 1] && L.A.cols[j] < L.n_owned)
          ++j;
        off[i] = j;
      }
      const int rc = pmgx_csr_create(ctx, L.n_owned, L.n_ghost, L.A.ptr.data(), off.data(), L.A.cols.data(),
                                     L.A.vals.data(), D.halo, &D.A);
      if (rc != PMGX_OK)
        return rc;
      D.own_A = true;
      const size_t nt = (size_t)L.n_owned + L.n_ghost;
      for (auto* buf : {&D.x, &D.b, &D.x2, &D.r2})
      {
        buf->alloc(nt);
        if (nt > 0)
          PMGX_CUDA(cudaMemsetAsync(buf->p, 0, nt * sizeof(double), ctx->stream));
      }
    }
    {
      const int rc = pmgx_cheb_create(ctx, L.n_owned, L.n_ghost, 0.1 * L.lmax, L.lmax, &D.sm);
      if (rc != PMGX_OK)
        return rc;
      // a coarsest level that could not be inverted densely is smoothed harder instead
      D.sm->max_iter = (last && !L.dense) ? 4 * nu : (l == 0 ? nu : nu_coarse);
      D.sm->fuse = l >= fuse_from;
    }
    // level 0's smoother streams the matrix with FP32 values and 16-bit column deltas (PMGX_AMG_LP=0: the FP64
    // matrix)
    if (l == 0 && !last && use_lp)
      D.A_lp = pmgx::make_lp(static_cast<pmgx::CsrOperator*>(D.A));
    D.nnz_p = L.P.nnz();
    if (!last)
    {
      // the transfers are smoothed with the full rows of A and carry its stored zeros as well (level 0's most)
      D.P.upload(pmgx::amg::drop_stored_zeros(L.P), ctx->stream);
      D.R.upload(pmgx::amg::drop_stored_zeros(L.R), ctx->stream);
    }
    else if (L.dense)
    {
      D.dense = true;
      D.n_global = (int)L.n_global;
      D.inv.upload(L.inv_rows.data(), L.inv_rows.size(), ctx->stream);
      const int n_gather = (int)L.n_global - L.n_owned;
      if (!L.replicated)
        D.gather = pmgx::make_halo(ctx, L.n_owned, n_gather, L.gather_plan);
      const size_t nt = (size_t)L.n_owned + std::max(L.n_ghost, n_gather);
      D.b.alloc(nt);
      if (nt > 0)
        PMGX_CUDA(cudaMemsetAsync(D.b.p, 0, nt * sizeof(double), ctx->stream));
    }
  }
  PMGX_CUDA(cudaStreamSynchronize(ctx->stream));

  pmgx_coarse* cs = nullptr;
  const int rc = pmgx_coarse_create(ctx, M->lv[0].A, max_iter, rtol, &cs); // PCG on the matrix without stored zeros too
  if (rc != PMGX_OK)
    return rc;
  cs->M = M.release();
  cs->check_every = 1; // an iteration costs ~0.7 ms, a host look at r.M^-1 r ~10 us
  if (const char* e = getenv("PMGX_COARSE_CHECK_EVERY"))
    cs->check_every = std::max(atoi(e), 1);
  *out = cs;
  PMGX_API_END
}

int pmgx_coarse_num_levels(pmgx_coarse* cs)
{
  if (!cs)
    return -1;
  return cs->M ? (int)static_cast<AmgPrecond*>(cs->M)->lv.size() : 1;
}

int pmgx_coarse_level_info(pmgx_coarse* cs, int level, long long* out_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(cs && out_h && level >= 0 && level < pmgx_coarse_num_levels(cs), "coarse_level_info: bad arguments");
  if (!cs->M)
  {
    out_h[0] = cs->A->n_owned;
    out_h[1] = pmgx_csr_nnz(cs->A);
    out_h[2] = cs->A->n_ghost;
    out_h[3] = 0;
    out_h[4] = 0;
  }
  else
  {
    const AmgPrecond::Lv& L = static_cast<AmgPrecond*>(cs->M)->lv[level];
    out_h[0] = L.n_owned;
    out_h[1] = L.nnz;
    out_h[2] = L.n_ghost;
    out_h[3] = L.dense ? 1 : 0;
    out_h[4] = L.nnz_p;
  }
  PMGX_API_END
}

int pmgx_coarse_apply_preconditioner(pmgx_coarse* cs, const double* r, double* u)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(cs && r && u && r != u, "coarse_apply_preconditioner: bad arguments");
  PMGX_CUDA(cudaSetDevice(cs->ctx->device));
  if (cs->M)
    cs->M->apply(r, u);
  else
    pmgx::vec::pointwise_mult(cs->ctx, u, r, cs->A->diag_inv.p, cs->A->n_owned);
  PMGX_API_END
}
}
