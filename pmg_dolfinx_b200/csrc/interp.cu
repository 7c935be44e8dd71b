// p-level prolongation / restriction as batched element-local sum-factorised kernels
// (north_star item 4).  Replaces interpolate_Q1Q2 / interpolate_Q2Q1 and Interpolator<T>
// (src/interpolate.hpp:21-87,93-329).
//
// Design (not a port of the per-cell CSR walk by one thread): a thread owns one fine z-index k
// of one cell.  The dofmap rows of the CTA's cells are staged in shared memory with coalesced
// loads; the z pass reads the coarse values (prolongation) or writes partial sums (restriction)
// across threads, the y and x passes are register FMAs against the 1-D interpolation table,
// which is a __grid_constant__ kernel parameter (constant-bank operands).  Every fine dof has a
// unique writer cell (quirk Q11: the reference lets several cells overwrite shared dofs with
// equal values), which halves the store traffic and lets u += P u_c be formed in the store.
// Cell lists live on the device (no per-call allocation, quirk Q10) and the fine-dof
// multiplicity is computed on the device.
#include "common.hpp"
#include "operator.hpp"

#include <cmath>
#include <cstring>
#include <type_traits>

namespace pmgx
{
namespace
{
struct InterpTab
{
  double m[(PMGX_MAX_DEGREE + 1) * (PMGX_MAX_DEGREE + 1)]; // M1[f * NC + c] = l^c_c(x^f_f)
};

// threads per CTA: the largest of {128, 64, 32} whose staged dofmap rows (+ the restriction's
// partial sums) stay below the 48 KB static shared-memory limit
template <int NC, int NF>
struct XferCfg
{
  static constexpr int bytes(int tpb)
  {
    const int cpb = tpb / NF;
    return cpb * (NC * NC * NC + NF * NF * NF) * 4 + cpb * NF * NC * NC * 8;
  }
  static constexpr int tpb = bytes(128) <= 46 * 1024 ? 128 : (bytes(64) <= 46 * 1024 ? 64 : 32);
  static constexpr int cpb = tpb / NF;
};

__global__ void k_count_mult(const int32_t* __restrict__ dm, long long total, double* __restrict__ mult)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nth)
    atomicAdd(&mult[dm[t]], 1.0);
}
__global__ void k_invert_mult(double* __restrict__ m, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
    m[i] = m[i] > 0.0 ? 1.0 / m[i] : 0.0;
}

// first list position that touches each fine dof ...
__global__ void k_first_toucher(const int32_t* __restrict__ dm_f, const int32_t* __restrict__ cells,
                                int nf3, long long total, int32_t* __restrict__ first)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nth)
  {
    const long long pos = t / nf3;
    const int j = (int)(t - pos * nf3);
    atomicMin(&first[dm_f[(long long)cells[pos] * nf3 + j]], (int32_t)pos);
  }
}
// ... becomes one writer bit per (list position, local fine dof)
__global__ void k_writer_mask(const int32_t* __restrict__ dm_f, const int32_t* __restrict__ cells,
                              const int32_t* __restrict__ first, int nf3, int words, long long n_list,
                              uint32_t* __restrict__ mask)
{
  const long long total = n_list * words;
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nth)
  {
    const long long pos = t / words;
    const int w = (int)(t - pos * words);
    uint32_t bits = 0;
    for (int b = 0; b < 32 && w * 32 + b < nf3; ++b)
      if (first[dm_f[(long long)cells[pos] * nf3 + w * 32 + b]] == (int32_t)pos)
        bits |= 1u << b;
    mask[t] = bits;
  }
}

// Prolongation: fine[dofs_f[j]] (=|+=) sum_k M[j,k] coarse[dofs_c[k]]   (src/interpolate.hpp:21-45;
// ADD folds the u += du of src/pmg.hpp:129, owned dofs only).
template <int NC, int NF, bool ADD>
__global__ void __launch_bounds__(XferCfg<NC, NF>::tpb)
k_prolong(const __grid_constant__ InterpTab tab, const int32_t* __restrict__ cells, int first, int count,
          const int32_t* __restrict__ dm_c, const int32_t* __restrict__ dm_f,
          const uint32_t* __restrict__ wmask, const double* __restrict__ xc, double* __restrict__ xf,
          int n_owned_f)
{
  constexpr int TPB = XferCfg<NC, NF>::tpb, CPB = XferCfg<NC, NF>::cpb;
  constexpr int NC3 = NC * NC * NC, NF3 = NF * NF * NF, W = (NF3 + 31) / 32;
  __shared__ int32_t s_c[CPB * NC3];
  __shared__ int32_t s_f[CPB * NF3]; // ~d when this cell is not the writer of d
  const int tid = threadIdx.x;
  const int cell0 = blockIdx.x * CPB;
  for (int idx = tid; idx < CPB * NC3; idx += TPB)
  {
    const int c = idx / NC3, j = idx - c * NC3;
    s_c[idx] = cell0 + c < count ? dm_c[(long long)cells[first + cell0 + c] * NC3 + j] : 0;
  }
  for (int idx = tid; idx < CPB * NF3; idx += TPB)
  {
    const int c = idx / NF3, j = idx - c * NF3;
    int32_t d = 0;
    if (cell0 + c < count)
    {
      d = dm_f[(long long)cells[first + cell0 + c] * NF3 + j];
      const uint32_t bits = wmask[(long long)(first + cell0 + c) * W + (j >> 5)];
      if (!((bits >> (j & 31)) & 1u))
        d = ~d;
    }
    s_f[idx] = d;
  }
  __syncthreads();
  const int c = tid / NF, k = tid - c * NF;
  if (c >= CPB || cell0 + c >= count)
    return;
  double mk[NC];
#pragma unroll
  for (int cz = 0; cz < NC; ++cz)
    mk[cz] = tab.m[k * NC + cz];
  // all global loads of the thread are issued before any arithmetic (the kernel is latency-bound:
  // ncu long_scoreboard 25 stalls per issue with the loads interleaved): NC^3 coarse values ...
  const int32_t* sc = s_c + c * NC3;
  const int32_t* sf = s_f + c * NF3 + k;
  double cv[NC3];
#pragma unroll
  for (int t = 0; t < NC3; ++t)
    cv[t] = xc[sc[t]];
  // ... and, when adding, the NF^2 fine values this thread owns
  double xo[ADD ? NF * NF : 1];
  if (ADD)
  {
#pragma unroll
    for (int t = 0; t < NF * NF; ++t)
    {
      const int32_t d = sf[t * NF];
      xo[t] = (d >= 0 && d < n_owned_f) ? xf[d] : 0.0;
    }
  }
  // z pass: v[ix][iy] = sum_cz M[k][cz] xc[ix][iy][cz]
  double v[NC][NC];
#pragma unroll
  for (int ix = 0; ix < NC; ++ix)
#pragma unroll
    for (int iy = 0; iy < NC; ++iy)
    {
      double s = 0.0;
#pragma unroll
      for (int cz = 0; cz < NC; ++cz)
        s = fma(mk[cz], cv[(ix * NC + iy) * NC + cz], s);
      v[ix][iy] = s;
    }
  // y pass: w[ix][fy] = sum_iy M[fy][iy] v[ix][iy]
  double w[NC][NF];
#pragma unroll
  for (int ix = 0; ix < NC; ++ix)
#pragma unroll
    for (int fy = 0; fy < NF; ++fy)
    {
      double s = 0.0;
#pragma unroll
      for (int iy = 0; iy < NC; ++iy)
        s = fma(tab.m[fy * NC + iy], v[ix][iy], s);
      w[ix][fy] = s;
    }
  // x pass + store by the unique writer
#pragma unroll
  for (int fx = 0; fx < NF; ++fx)
#pragma unroll
    for (int fy = 0; fy < NF; ++fy)
    {
      double s = 0.0;
#pragma unroll
      for (int ix = 0; ix < NC; ++ix)
        s = fma(tab.m[fx * NC + ix], w[ix][fy], s);
      const int32_t d = sf[(fx * NF + fy) * NF];
      if (d >= 0)
      {
        if (ADD)
        {
          if (d < n_owned_f)
            xf[d] = s * 1.0 + xo[fx * NF + fy];
        }
        else
          xf[d] = s;
      }
    }
}

// Restriction: coarse[dofs_c[j]] += sum_k M[k,j] (fine[d_k] - sub[d_k]) / mult[d_k]
// (atomics; src/interpolate.hpp:60-87).  sub (may be null) is subtracted on owned fine dofs only:
// it folds the smoother's last r -= q into the gather.
template <int NC, int NF>
__global__ void __launch_bounds__(XferCfg<NC, NF>::tpb)
k_restrict(const __grid_constant__ InterpTab tab, const int32_t* __restrict__ cells, int first, int count,
           const int32_t* __restrict__ dm_c, const int32_t* __restrict__ dm_f, const double* __restrict__ xf,
           const double* __restrict__ sub, int n_owned_f, const double* __restrict__ inv_mult,
           double* __restrict__ xc)
{
  constexpr int TPB = XferCfg<NC, NF>::tpb, CPB = XferCfg<NC, NF>::cpb;
  constexpr int NC2 = NC * NC, NC3 = NC2 * NC, NF3 = NF * NF * NF;
  __shared__ int32_t s_c[CPB * NC3];
  __shared__ int32_t s_f[CPB * NF3];
  __shared__ double s_v[CPB * NF * NC2];
  const int tid = threadIdx.x;
  const int cell0 = blockIdx.x * CPB;
  for (int idx = tid; idx < CPB * NC3; idx += TPB)
  {
    const int c = idx / NC3, j = idx - c * NC3;
    s_c[idx] = cell0 + c < count ? dm_c[(long long)cells[first + cell0 + c] * NC3 + j] : 0;
  }
  for (int idx = tid; idx < CPB * NF3; idx += TPB)
  {
    const int c = idx / NF3, j = idx - c * NF3;
    s_f[idx] = cell0 + c < count ? dm_f[(long long)cells[first + cell0 + c] * NF3 + j] : 0;
  }
  __syncthreads();
  const int c = tid / NF, k = tid - c * NF;
  if (c < CPB)
  {
    const bool active = cell0 + c < count;
    // transposed x pass: w[ix][fy] = sum_fx M[fx][ix] val[fx][fy]
    double w[NC][NF];
#pragma unroll
    for (int ix = 0; ix < NC; ++ix)
#pragma unroll
      for (int fy = 0; fy < NF; ++fy)
        w[ix][fy] = 0.0;
    const int32_t* sf = s_f + c * NF3 + k;
    if (active)
    {
      // gathers run one fx-slice ahead of the arithmetic (latency-bound kernel: 3 NF loads in flight)
      double fv[2][NF], sv2[2][NF], mv[2][NF];
      auto load_slice = [&](int fx, int b)
      {
#pragma unroll
        for (int fy = 0; fy < NF; ++fy)
        {
          const int32_t d = sf[(fx * NF + fy) * NF];
          fv[b][fy] = xf[d];
          sv2[b][fy] = (sub != nullptr && d < n_owned_f) ? sub[d] : 0.0;
          mv[b][fy] = inv_mult[d];
        }
      };
      load_slice(0, 0);
#pragma unroll
      for (int fx = 0; fx < NF; ++fx)
      {
        if (fx + 1 < NF)
          load_slice(fx + 1, (fx + 1) & 1);
#pragma unroll
        for (int fy = 0; fy < NF; ++fy)
        {
          double val = fv[fx & 1][fy];
          if (sub != nullptr)
            val = sv2[fx & 1][fy] * (-1.0) + val; // ghost entries carry 0 here: x - 0 is exact
          val *= mv[fx & 1][fy]; // src/interpolate.hpp:82
#pragma unroll
          for (int ix = 0; ix < NC; ++ix)
            w[ix][fy] = fma(tab.m[fx * NC + ix], val, w[ix][fy]);
        }
      }
    }
    // transposed y pass: v[ix][iy] = sum_fy M[fy][iy] w[ix][fy]; handed to the z pass through smem
    double* sv = s_v + (c * NF + k) * NC2;
#pragma unroll
    for (int ix = 0; ix < NC; ++ix)
#pragma unroll
      for (int iy = 0; iy < NC; ++iy)
      {
        double s = 0.0;
#pragma unroll
        for (int fy = 0; fy < NF; ++fy)
          s = fma(tab.m[fy * NC + iy], w[ix][fy], s);
        sv[ix * NC + iy] = s;
      }
  }
  __syncthreads();
  // transposed z pass: coarse (ix,iy,cz) += sum_k M[k][cz] v_k[ix][iy]; one atomic per coarse dof and cell
  for (int idx = tid; idx < CPB * NC3; idx += TPB)
  {
    const int cc = idx / NC3, j = idx - cc * NC3;
    if (cell0 + cc >= count)
      break;
    const int ixy = j / NC, cz = j - ixy * NC;
    double s = 0.0;
#pragma unroll
    for (int kk = 0; kk < NF; ++kk)
      s = fma(tab.m[kk * NC + cz], s_v[(cc * NF + kk) * NC2 + ixy], s);
    atomicAdd(&xc[s_c[idx]], s);
  }
}

// x[idx] - sub[idx] into the send buffer is done by the halo (halo_fwd_begin with sub)
} // namespace
} // namespace pmgx

struct pmgx_interp
{
  pmgx_ctx* ctx = nullptr;
  int pc = 0, pf = 0, n_cells = 0, n_l = 0, n_b = 0;
  int n_coarse_total = 0, n_fine_total = 0;
  const int32_t* dm_c = nullptr; // borrowed device dofmaps (src/interpolate.hpp:322-323)
  const int32_t* dm_f = nullptr;
  pmgx_halo* halo_c = nullptr;
  pmgx_halo* halo_f = nullptr;
  pmgx::DevBuf<int32_t> cells;   // lcells then bcells
  pmgx::DevBuf<uint32_t> wmask;  // [n_list][ceil(nf^3/32)] unique-writer bits
  pmgx::DevBuf<double> inv_mult; // 1 / multiplicity of fine dofs
  pmgx::InterpTab tab;
};

namespace pmgx
{
namespace
{
template <int NC, int NF>
void launch_prolong(pmgx_interp* it, cudaStream_t st, int first, int count, const double* xc, double* xf, bool add)
{
  if (count <= 0)
    return;
  pmgx_ctx* c = it->ctx;
  using C = XferCfg<NC, NF>;
  const int grid = (count + C::cpb - 1) / C::cpb;
  const int n_owned_f = it->halo_f ? it->halo_f->n_owned : it->n_fine_total;
  if (add)
    k_prolong<NC, NF, true><<<grid, C::tpb, 0, st>>>(it->tab, it->cells.p, first, count, it->dm_c, it->dm_f,
                                                           it->wmask.p, xc, xf, n_owned_f);
  else
    k_prolong<NC, NF, false><<<grid, C::tpb, 0, st>>>(it->tab, it->cells.p, first, count, it->dm_c, it->dm_f,
                                                            it->wmask.p, xc, xf, n_owned_f);
  check_launch("k_prolong");
  count_launch(c);
}

template <int NC, int NF>
void launch_restrict(pmgx_interp* it, cudaStream_t st, int first, int count, const double* xf, const double* sub,
                     double* xc)
{
  if (count <= 0)
    return;
  pmgx_ctx* c = it->ctx;
  using C = XferCfg<NC, NF>;
  const int grid = (count + C::cpb - 1) / C::cpb;
  const int n_owned_f = it->halo_f ? it->halo_f->n_owned : it->n_fine_total;
  k_restrict<NC, NF><<<grid, C::tpb, 0, st>>>(it->tab, it->cells.p, first, count, it->dm_c, it->dm_f, xf, sub,
                                                     n_owned_f, it->inv_mult.p, xc);
  check_launch("k_restrict");
  count_launch(c);
}

// dispatch on (coarse, fine) nodes per direction; pc <= pf
template <int NF, typename F>
void dispatch_nc(int nc, F&& f)
{
  switch (nc)
  {
  case 2: f(std::integral_constant<int, 2>{}); break;
  case 3: if constexpr (NF >= 3) f(std::integral_constant<int, 3>{}); break;
  case 4: if constexpr (NF >= 4) f(std::integral_constant<int, 4>{}); break;
  case 5: if constexpr (NF >= 5) f(std::integral_constant<int, 5>{}); break;
  case 6: if constexpr (NF >= 6) f(std::integral_constant<int, 6>{}); break;
  case 7: if constexpr (NF >= 7) f(std::integral_constant<int, 7>{}); break;
  case 8: if constexpr (NF >= 8) f(std::integral_constant<int, 8>{}); break;
  case 9: if constexpr (NF >= 9) f(std::integral_constant<int, 9>{}); break;
  default: break;
  }
}
template <typename F>
void dispatch(int nc, int nf, F&& f)
{
  switch (nf)
  {
  case 2: dispatch_nc<2>(nc, [&](auto NC) { f(NC, std::integral_constant<int, 2>{}); }); break;
  case 3: dispatch_nc<3>(nc, [&](auto NC) { f(NC, std::integral_constant<int, 3>{}); }); break;
  case 4: dispatch_nc<4>(nc, [&](auto NC) { f(NC, std::integral_constant<int, 4>{}); }); break;
  case 5: dispatch_nc<5>(nc, [&](auto NC) { f(NC, std::integral_constant<int, 5>{}); }); break;
  case 6: dispatch_nc<6>(nc, [&](auto NC) { f(NC, std::integral_constant<int, 6>{}); }); break;
  case 7: dispatch_nc<7>(nc, [&](auto NC) { f(NC, std::integral_constant<int, 7>{}); }); break;
  case 8: dispatch_nc<8>(nc, [&](auto NC) { f(NC, std::integral_constant<int, 8>{}); }); break;
  case 9: dispatch_nc<9>(nc, [&](auto NC) { f(NC, std::integral_constant<int, 9>{}); }); break;
  default: break;
  }
}
} // namespace

// interpolate (src/interpolate.hpp:185-239); add: fine += P coarse on owned fine dofs.
// Interior cells run on the compute stream while the coarse halo is in flight (:202-208); the
// boundary cells (:217-227) are enqueued right behind the exchange on the halo stream (every
// fine dof has one writer, so the two launches never touch the same entry).
void interp_prolong(pmgx_interp* it, double* coarse, double* fine, bool add)
{
  pmgx_ctx* c = it->ctx;
  PMGX_CUDA(cudaSetDevice(c->device));
  if (it->halo_c)
    halo_fwd_begin(it->halo_c, coarse);
  cudaStream_t bs = halo_stream(it->halo_c, c);
  dispatch(it->pc + 1, it->pf + 1, [&](auto NC, auto NF)
           { launch_prolong<NC(), NF()>(it, c->stream, 0, it->n_l, coarse, fine, add); });
  dispatch(it->pc + 1, it->pf + 1, [&](auto NC, auto NF)
           { launch_prolong<NC(), NF()>(it, bs, it->n_l, it->n_b, coarse, fine, add); });
  if (it->halo_c)
    halo_fwd_end(it->halo_c, coarse);
}

// reverse_interpolate (src/interpolate.hpp:245-303) of fine - sub (sub may be null).  The output
// is zeroed (:270) before the exchange starts so that both launches may accumulate into it.
void interp_restrict(pmgx_interp* it, double* fine, const double* sub, double* coarse)
{
  pmgx_ctx* c = it->ctx;
  PMGX_CUDA(cudaSetDevice(c->device));
  vec::set(c, coarse, it->n_coarse_total, 0.0);
  if (it->halo_f)
    halo_fwd_begin(it->halo_f, fine, sub);                                           // :264
  cudaStream_t bs = halo_stream(it->halo_f, c);
  dispatch(it->pc + 1, it->pf + 1, [&](auto NC, auto NF)
           { launch_restrict<NC(), NF()>(it, c->stream, 0, it->n_l, fine, sub, coarse); });
  dispatch(it->pc + 1, it->pf + 1, [&](auto NC, auto NF)
           { launch_restrict<NC(), NF()>(it, bs, it->n_l, it->n_b, fine, sub, coarse); });
  if (it->halo_f)
    halo_fwd_end(it->halo_f, fine);                                                  // :281
}
} // namespace pmgx

extern "C"
{
int pmgx_interp_create(pmgx_ctx* ctx, int degree_coarse, int degree_fine, int n_cells,
                       const int32_t* dofmap_coarse, const int32_t* dofmap_fine, int n_coarse_total,
                       int n_fine_total, const int32_t* lcells_h, int n_lcells,
                       const int32_t* bcells_h, int n_bcells, pmgx_halo* halo_c, pmgx_halo* halo_f,
                       pmgx_interp** out)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(ctx && out, "interp_create: null ctx/out");
  PMGX_REQUIRE(degree_coarse >= 1 && degree_fine <= PMGX_MAX_DEGREE && degree_coarse <= degree_fine,
               "Unsupported degrees %d -> %d", degree_coarse, degree_fine);
  PMGX_REQUIRE(n_cells >= 0 && n_lcells >= 0 && n_bcells >= 0 && n_lcells + n_bcells <= n_cells,
               "interp_create: inconsistent cell counts");
  PMGX_REQUIRE(n_cells == 0 || (dofmap_coarse && dofmap_fine), "interp_create: null dofmap");
  PMGX_REQUIRE(!halo_f || halo_f->n_owned + halo_f->n_ghost == n_fine_total,
               "interp_create: fine halo does not match the fine vector layout");
  PMGX_REQUIRE(!halo_c || halo_c->n_owned + halo_c->n_ghost == n_coarse_total,
               "interp_create: coarse halo does not match the coarse vector layout");
  PMGX_CUDA(cudaSetDevice(ctx->device));
  std::unique_ptr<pmgx_interp> it(new pmgx_interp());
  it->ctx = ctx;
  it->pc = degree_coarse;
  it->pf = degree_fine;
  it->n_cells = n_cells;
  it->n_l = n_lcells;
  it->n_b = n_bcells;
  it->n_coarse_total = n_coarse_total;
  it->n_fine_total = n_fine_total;
  it->dm_c = dofmap_coarse;
  it->dm_f = dofmap_fine;
  it->halo_c = halo_c;
  it->halo_f = halo_f;
  const int n_list = n_lcells + n_bcells;
  std::vector<int32_t> cl((size_t)n_list);
  for (int i = 0; i < n_lcells; ++i)
    cl[i] = lcells_h[i];
  for (int i = 0; i < n_bcells; ++i)
    cl[n_lcells + i] = bcells_h[i];
  for (int32_t v : cl)
    PMGX_REQUIRE(v >= 0 && v < n_cells, "interp_create: cell index out of range");
  it->cells.upload(cl.data(), cl.size(), ctx->stream);
  std::vector<double> M;
  pmgx::gll_interp_matrix(degree_coarse, degree_fine, M);
  std::memset(&it->tab, 0, sizeof(it->tab));
  for (size_t i = 0; i < M.size(); ++i) // the reference drops |v| <= 1e-12 when compressing (interpolate.hpp:120-128)
    it->tab.m[i] = std::fabs(M[i]) <= 1e-12 ? 0.0 : M[i];
  const int nf = degree_fine + 1, nf3 = nf * nf * nf;
  auto sgrid = [&](long long total)
  { return (int)std::max<long long>(1, std::min<long long>((total + 255) / 256, ctx->num_sms * 32)); };
  // multiplicity over the whole fine dofmap (all local + ghost cells, :172-178)
  it->inv_mult.alloc((size_t)n_fine_total);
  if (n_fine_total > 0)
  {
    PMGX_CUDA(cudaMemsetAsync(it->inv_mult.p, 0, (size_t)n_fine_total * sizeof(double), ctx->stream));
    const long long total = (long long)n_cells * nf3;
    if (total > 0)
    {
      pmgx::k_count_mult<<<sgrid(total), 256, 0, ctx->stream>>>(dofmap_fine, total, it->inv_mult.p);
      pmgx::check_launch("k_count_mult");
    }
    pmgx::k_invert_mult<<<(n_fine_total + 255) / 256, 256, 0, ctx->stream>>>(it->inv_mult.p, n_fine_total);
    pmgx::check_launch("k_invert_mult");
    pmgx::count_launch(ctx, 2);
  }
  // unique writer of every fine dof: the first cell of the launch list that touches it
  const int words = (nf3 + 31) / 32;
  it->wmask.alloc((size_t)std::max(1, n_list) * words);
  if (n_list > 0 && n_fine_total > 0)
  {
    pmgx::DevBuf<int32_t> first;
    first.alloc((size_t)n_fine_total);
    PMGX_CUDA(cudaMemsetAsync(first.p, 0x7f, (size_t)n_fine_total * sizeof(int32_t), ctx->stream));
    const long long total = (long long)n_list * nf3;
    pmgx::k_first_toucher<<<sgrid(total), 256, 0, ctx->stream>>>(dofmap_fine, it->cells.p, nf3, total, first.p);
    pmgx::check_launch("k_first_toucher");
    pmgx::k_writer_mask<<<sgrid((long long)n_list * words), 256, 0, ctx->stream>>>(
        dofmap_fine, it->cells.p, first.p, nf3, words, n_list, it->wmask.p);
    pmgx::check_launch("k_writer_mask");
    pmgx::count_launch(ctx, 2);
    PMGX_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  PMGX_CUDA(cudaStreamSynchronize(ctx->stream));
  *out = it.release();
  PMGX_API_END
}

int pmgx_interp_prolong(pmgx_interp* it, double* coarse, double* fine)
{
  PMGX_API_BEGIN
  // a rank without cells has zero-length vectors, whose device pointers may be null
  PMGX_REQUIRE(it && (coarse || it->n_coarse_total == 0) && (fine || it->n_fine_total == 0),
               "interp_prolong: null argument");
  pmgx::interp_prolong(it, coarse, fine, false);
  PMGX_API_END
}

int pmgx_interp_restrict(pmgx_interp* it, double* fine, double* coarse)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(it && (coarse || it->n_coarse_total == 0) && (fine || it->n_fine_total == 0),
               "interp_restrict: null argument");
  pmgx::interp_restrict(it, fine, nullptr, coarse);
  PMGX_API_END
}

int pmgx_interp_destroy(pmgx_interp* it)
{
  PMGX_API_BEGIN
  if (it)
  {
    cudaSetDevice(it->ctx->device);
    cudaStreamSynchronize(it->ctx->stream);
    delete it;
  }
  PMGX_API_END
}
}
