// Exterior-facet Dirichlet marker on the device: what the reference drivers obtain on the host from
// mesh::exterior_facet_indices + fem::locate_dofs_topological (examples/pmg/main.cpp:173-185,
// examples/cg/main.cpp:150-158) -- SURVEY 8f-2 "BC marker generation".
//
// A facet is exterior iff it belongs to exactly one cell.  Every rank only sees its owned + ghost cells, so
// a facet on the outer rim of the ghost layer LOOKS exterior locally; but a facet that touches an OWNED dof
// has all of its cells here (every cell containing an owned dof is local, src/mesh.hpp:25-46), so the local
// count is exact for every owned dof.  Hence: count facets locally (sort of the 4 sorted vertex ids), mark
// the (P+1)^2 dofs of every facet seen once, then let the owners overwrite the ghost entries with one
// forward halo update.
#include "common.hpp"
#include "operator.hpp"

#include <thrust/device_ptr.h>
#include <thrust/execution_policy.h>
#include <thrust/sequence.h>
#include <thrust/sort.h>

namespace pmgx
{
namespace
{
// facet q of the reference hex: direction d = q / 2 fixed at side s = q % 2; vertex k = 4a + 2b + c
__device__ __forceinline__ void facet_vertices(const int32_t* __restrict__ gd, int q, unsigned int v[4])
{
  const int d = q >> 1, s = q & 1;
  int t = 0;
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b)
    {
      const int abc[3] = {d == 0 ? s : a, d == 1 ? s : (d == 0 ? a : b), d == 2 ? s : b};
      v[t++] = (unsigned int)gd[4 * abc[0] + 2 * abc[1] + abc[2]];
    }
  // sort 4 (network)
#define PMGX_CSWAP(i, j)                                                                           \
  if (v[i] > v[j])                                                                                 \
  {                                                                                                \
    const unsigned int tmp = v[i];                                                                 \
    v[i] = v[j];                                                                                   \
    v[j] = tmp;                                                                                    \
  }
  PMGX_CSWAP(0, 1)
  PMGX_CSWAP(2, 3)
  PMGX_CSWAP(0, 2)
  PMGX_CSWAP(1, 3)
  PMGX_CSWAP(1, 2)
#undef PMGX_CSWAP
}

__global__ void k_facet_keys(long long n_facets, const int32_t* __restrict__ geom_dofmap,
                             unsigned long long* __restrict__ hi, unsigned long long* __restrict__ lo)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x; f < n_facets; f += nth)
  {
    unsigned int v[4];
    facet_vertices(geom_dofmap + (f / 6) * 8, (int)(f % 6), v);
    hi[f] = ((unsigned long long)v[0] << 32) | v[1];
    lo[f] = ((unsigned long long)v[2] << 32) | v[3];
  }
}

__global__ void k_gather_u64(long long n, const int32_t* __restrict__ idx, const unsigned long long* __restrict__ in,
                             unsigned long long* __restrict__ out)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += nth)
    out[i] = in[idx[i]];
}

// sorted position p holds facet idx[p]; it is exterior iff its key differs from both neighbours'.  All
// (P+1)^2 dofs of an exterior facet get mark 1.
__global__ void k_mark_exterior(long long n_facets, const int32_t* __restrict__ idx, const unsigned long long* __restrict__ hi,
                                const unsigned long long* __restrict__ lo, int n, const int32_t* __restrict__ dofmap,
                                double* __restrict__ mark)
{
  const int n2 = n * n, n3 = n2 * n;
  const long long total = n_facets * n2;
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nth)
  {
    const long long p = t / n2;
    const int r = (int)(t - p * n2);
    const int f = idx[p];
    bool once = true;
    if (p > 0)
    {
      const int g = idx[p - 1];
      once = once && !(hi[g] == hi[f] && lo[g] == lo[f]);
    }
    if (p + 1 < n_facets)
    {
      const int g = idx[p + 1];
      once = once && !(hi[g] == hi[f] && lo[g] == lo[f]);
    }
    if (!once)
      continue;
    const int cell = f / 6, q = f % 6, d = q >> 1, s = (q & 1) * (n - 1);
    const int u = r / n, w = r - u * n;
    const int ix = d == 0 ? s : u, iy = d == 1 ? s : (d == 0 ? u : w), iz = d == 2 ? s : w;
    mark[dofmap[(long long)cell * n3 + (ix * n + iy) * n + iz]] = 1.0;
  }
}

__global__ void k_to_marker(int n, const double* __restrict__ mark, int8_t* __restrict__ out)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
    out[i] = mark[i] != 0.0 ? 1 : 0;
}
} // namespace
} // namespace pmgx

extern "C" int pmgx_bc_marker_exterior(pmgx_ctx* ctx, int degree, int n_cells, const int32_t* geom_dofmap,
                                       const int32_t* dofmap, int n_owned, int n_ghost, pmgx_halo* halo,
                                       int8_t* marker_out)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(ctx && degree >= 1 && degree <= PMGX_MAX_DEGREE, "bc_marker_exterior: bad arguments");
  PMGX_REQUIRE(n_cells >= 0 && n_owned >= 0 && n_ghost >= 0 && (long long)n_cells * 6 < (1ll << 31),
               "bc_marker_exterior: bad sizes");
  // a rank without cells has a zero-length marker, whose device pointer may be null
  PMGX_REQUIRE(marker_out || n_owned + n_ghost == 0, "bc_marker_exterior: null marker");
  PMGX_REQUIRE(n_cells == 0 || (geom_dofmap && dofmap), "bc_marker_exterior: null array");
  PMGX_REQUIRE(!halo || (halo->n_owned == n_owned && halo->n_ghost == n_ghost), "bc_marker_exterior: halo does not match the layout");
  PMGX_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int nt = n_owned + n_ghost;
  const long long nf = (long long)n_cells * 6;
  pmgx::DevBuf<double> mark;
  mark.alloc((size_t)std::max(nt, 1));
  PMGX_CUDA(cudaMemsetAsync(mark.p, 0, (size_t)std::max(nt, 1) * sizeof(double), st));
  if (nf > 0)
  {
    pmgx::DevBuf<unsigned long long> hi, lo, key;
    pmgx::DevBuf<int32_t> idx;
    hi.alloc((size_t)nf);
    lo.alloc((size_t)nf);
    key.alloc((size_t)nf);
    idx.alloc((size_t)nf);
    const int grid = (int)std::min<long long>((nf + 255) / 256, (long long)ctx->num_sms * 32);
    pmgx::k_facet_keys<<<grid, 256, 0, st>>>(nf, geom_dofmap, hi.p, lo.p);
    pmgx::check_launch("k_facet_keys");
    auto pol = thrust::cuda::par.on(st);
    thrust::device_ptr<int32_t> ip(idx.p);
    thrust::device_ptr<unsigned long long> kp(key.p);
    thrust::sequence(pol, ip, ip + nf);
    // lexicographic (hi, lo) order: sort by lo, then stably by hi
    PMGX_CUDA(cudaMemcpyAsync(key.p, lo.p, (size_t)nf * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, st));
    thrust::sort_by_key(pol, kp, kp + nf, ip);
    pmgx::k_gather_u64<<<grid, 256, 0, st>>>(nf, idx.p, hi.p, key.p);
    pmgx::check_launch("k_gather_u64");
    thrust::stable_sort_by_key(pol, kp, kp + nf, ip);
    const int n = degree + 1;
    const long long total = nf * n * n;
    const int g2 = (int)std::min<long long>((total + 255) / 256, (long long)ctx->num_sms * 32);
    pmgx::k_mark_exterior<<<g2, 256, 0, st>>>(nf, idx.p, hi.p, lo.p, n, dofmap, mark.p);
    pmgx::check_launch("k_mark_exterior");
    pmgx::count_launch(ctx, 3);
    PMGX_CUDA(cudaStreamSynchronize(st));
  }
  if (halo)
  {
    pmgx::halo_fwd_begin(halo, mark.p); // the owners' values replace whatever the rim of the ghost layer suggested
    pmgx::halo_fwd_end(halo, mark.p);
  }
  if (nt > 0)
  {
    pmgx::k_to_marker<<<(nt + 255) / 256, 256, 0, st>>>(nt, mark.p, marker_out);
    pmgx::check_launch("k_to_marker");
    pmgx::count_launch(ctx);
  }
  PMGX_CUDA(cudaStreamSynchronize(st));
  PMGX_API_END
}
