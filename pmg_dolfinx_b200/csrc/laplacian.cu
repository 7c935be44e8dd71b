// Matrix-free hexahedral Laplacian for P1..P8 on sm_100a.
//
// Replaces (reference paths):
//   geometry_computation<T,P>   src/laplacian.hpp:22-113
//   stiffness_operator<T,P>     src/laplacian.hpp:143-278
//   MatFreeLaplacian<T>         src/laplacian.hpp:283-526
//   diagonal via assembled CSR  examples/pmg/main.cpp:274-279, src/csr.hpp:101-112
//
// Design (not a port): cells are re-laid-out at create time in launch order (lcells then
// bcells); the dofmap is snapshotted with the Dirichlet marker folded into the sign bit, so
// the apply never gathers bc_marker; G is stored component-major per batch of cells so that one
// (ix) plane of a batch is one contiguous cp.async.bulk transaction.  One apply kernel per degree
// and geometry, chosen in ApplyKernels<P> below:
//   k_apply_affine / _affine_shfl / _affine2   P1..P5, every cell affine: one geometry 6-vector per cell
//   k_apply_tma                                P1..P5, G streamed per quadrature point through a TMA ring
//   k_apply_affine_mma                         P6, P7: FP64 tensor cores, one warp per cell (laplacian_mma.cuh)
//   k_apply                                    P8: column kernel
// and, for PMGX_LAP_RECOMPUTE_G, a variant of each of the last three families that forms G at its points from the
// cell's vertices instead of reading it (no per-point geometry is stored).
// In the slab kernels (P1..P5) a thread owns one z-index of a cell and keeps the (ix,iy) slab of
// the element in registers: the x and y contractions are register FMAs against constant-memory
// derivative entries, only the z contraction crosses threads.
#include "common.hpp"
#include "operator.hpp"
#include "csr.hpp"

#include <thrust/device_ptr.h>
#include <thrust/execution_policy.h>
#include <thrust/reduce.h>
#include <thrust/sort.h>
#include <thrust/scan.h>

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <type_traits>

namespace pmgx
{
namespace
{
constexpr int MAXN = PMGX_MAX_DEGREE + 1;

// 1-D tables for every degree; index [P][...]
__constant__ double c_D[PMGX_MAX_DEGREE + 1][MAXN * MAXN]; // D[q*n+i] = l_i'(x_q)
__constant__ double c_pts[PMGX_MAX_DEGREE + 1][MAXN];
__constant__ double c_wts[PMGX_MAX_DEGREE + 1][MAXN];

__device__ __forceinline__ double ldg_stream(const double* p)
{
  // streamed exactly once per apply: ld.global.cs (evict-first) keeps the gathered /
  // scattered x and y lines resident in L2 instead of the one-shot G / dofmap stream
  return __ldcs(p);
}
__device__ __forceinline__ int ldg_stream_i32(const int* p) { return __ldcs(p); }


// How the operator-private arrays (BC-encoded dofmap, geometry factors) are laid out.  The
// reference keeps G private (src/laplacian.hpp:512), so the layout is free: it follows the
// thread mapping of the apply kernel so that every warp load is one aligned, contiguous run.
//   COLUMN: enc[p][n3], G[p][6][n3]                         (P6..P8: a warp or an (iy,iz) column per cell)
//   SLAB  : enc[batch][n2][SE], G[batch][n2][6][S]          (P1..P5: thread = iz slab)
//           batch = cpb consecutive cells of the launch list (cpb of the kernel that runs),
//           slot = cell_in_batch*n + iz, S / SE padded to 16-byte rows; lcells and bcells
//           batches are padded separately.
struct Lay
{
  int mode; // 0 COLUMN, 1 SLAB
  int n, n2, n3;
  int cpb, S, SE; // SE: slot stride of the int32 dofmap rows (multiple of 4 -> 16-byte rows)
  int n_l, nb_l;
  long long n_batches;
  __host__ __device__ long long enc_size() const { return mode == 0 ? 0 : n_batches * n2 * SE; }
  __host__ __device__ long long g_size() const { return mode == 0 ? 0 : n_batches * n2 * 6 * S; }
  __host__ __device__ long long enc_index(long long p, int a) const
  {
    if (mode == 0)
      return p * n3 + a;
    const long long pl = p < n_l ? p : p - n_l;
    const long long batch = (p < n_l ? 0 : nb_l) + pl / cpb;
    const int slot = (int)(pl % cpb) * n + a % n;
    return (batch * n2 + a / n) * SE + slot;
  }
  __host__ __device__ long long g_index(long long p, int comp, int q) const
  {
    if (mode == 0)
      return (p * 6 + comp) * n3 + q;
    const long long pl = p < n_l ? p : p - n_l;
    const long long batch = (p < n_l ? 0 : nb_l) + pl / cpb;
    const int slot = (int)(pl % cpb) * n + q % n;
    return ((batch * n2 + q / n) * 6 + comp) * S + slot;
  }
};

// ------------------------------------------------------------------ set-up kernels --
__global__ void k_encode_dofmap(const int32_t* __restrict__ dofmap, const int32_t* __restrict__ perm,
                                const int8_t* __restrict__ bc, int32_t* __restrict__ enc, int n3,
                                long long total, Lay lay)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nth)
  {
    const long long p = t / n3;
    const int a = (int)(t - p * n3);
    const int32_t d = dofmap[(long long)perm[p] * n3 + a];
    enc[lay.enc_index(p, a)] = bc[d] ? ~d : d;
  }
}

// ------------------------------------------------------- geometry of the trilinear hexahedron --
// J, K = adj(J), det J and G = s K K^T (6 unique entries xx,xy,xz,yy,yz,zz) for every path that forms G from the
// vertices without storing it (PMGX_LAP_RECOMPUTE_G).  Vertex order k = 4a + 2b + c (src/mesh.hpp:75-84).  The
// set-up paths go through jacobian_at; the apply kernels form J in the factored per-thread forms of
// TrilinearMonomials.  k_geometry and k_cell_geometry below keep their own copy of the same expressions: routed
// through these helpers, k_geometry's G changed in the last bit on perturbed meshes (different FMA contraction).

// J = sum_k x_k dphi_k(xi), the vertices read from xgeom through the cell's 8 geometry dofs gd
__device__ __forceinline__ void jacobian_at(const double* __restrict__ xgeom, const int32_t* __restrict__ gd,
                                            const double (&xi)[3], double (&J)[3][3])
{
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      J[i][j] = 0.0;
#pragma unroll
  for (int k = 0; k < 8; ++k)
  {
    const int a = (k >> 2) & 1, b = (k >> 1) & 1, c = k & 1;
    const double la = a ? xi[0] : 1.0 - xi[0], lb = b ? xi[1] : 1.0 - xi[1],
                 lc = c ? xi[2] : 1.0 - xi[2];
    const double da = a ? 1.0 : -1.0, db = b ? 1.0 : -1.0, dc = c ? 1.0 : -1.0;
    const double dphi[3] = {da * lb * lc, la * db * lc, la * lb * dc};
    const double* xv = xgeom + 3ll * gd[k];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j)
        J[i][j] += xv[i] * dphi[j];
  }
}

// K = adj(J) and det J; literal_detj: the expression of src/laplacian.hpp:97 (quirk Q17)
__device__ __forceinline__ double adjugate_det(const double (&J)[3][3], bool literal_detj, double (&K)[3][3])
{
  K[0][0] = J[1][1] * J[2][2] - J[1][2] * J[2][1];
  K[0][1] = -J[0][1] * J[2][2] + J[0][2] * J[2][1];
  K[0][2] = J[0][1] * J[1][2] - J[0][2] * J[1][1];
  K[1][0] = -J[1][0] * J[2][2] + J[1][2] * J[2][0];
  K[1][1] = J[0][0] * J[2][2] - J[0][2] * J[2][0];
  K[1][2] = -J[0][0] * J[1][2] + J[0][2] * J[1][0];
  K[2][0] = J[1][0] * J[2][1] - J[1][1] * J[2][0];
  K[2][1] = -J[0][0] * J[2][1] + J[0][1] * J[2][0];
  K[2][2] = J[0][0] * J[1][1] - J[0][1] * J[1][0];
  double detJ;
  if (literal_detj)
    detJ = J[0][0] * K[0][0] - J[1][0] * K[0][1] + J[0][2] * K[2][0];
  else
    detJ = J[0][0] * K[0][0] + J[0][1] * K[1][0] + J[0][2] * K[2][0];
  return detJ;
}

// g = s K K^T (s = w / det J)
__device__ __forceinline__ void g_from_adjugate(const double (&K)[3][3], double s, double (&g)[6])
{
  g[0] = (K[0][0] * K[0][0] + K[0][1] * K[0][1] + K[0][2] * K[0][2]) * s;
  g[1] = (K[1][0] * K[0][0] + K[1][1] * K[0][1] + K[1][2] * K[0][2]) * s;
  g[2] = (K[2][0] * K[0][0] + K[2][1] * K[0][1] + K[2][2] * K[0][2]) * s;
  g[3] = (K[1][0] * K[1][0] + K[1][1] * K[1][1] + K[1][2] * K[1][2]) * s;
  g[4] = (K[2][0] * K[1][0] + K[2][1] * K[1][1] + K[2][2] * K[1][2]) * s;
  g[5] = (K[2][0] * K[2][0] + K[2][1] * K[2][1] + K[2][2] * K[2][2]) * s;
}

// g = w K K^T / det J of the Jacobian J
__device__ __forceinline__ void g_from_jacobian(const double (&J)[3][3], bool literal_detj, double w, double (&g)[6])
{
  double K[3][3];
  const double detJ = adjugate_det(J, literal_detj, K);
  g_from_adjugate(K, w / detJ, g);
}

// The trilinear map in monomial form, x = a0 + a1 xi + a2 eta + a3 zeta + a4 xi eta + a5 xi zeta + a6 eta zeta
// + a7 xi eta zeta (m[0..6] = a1..a7, one 3-vector each), so that the Jacobian columns are
//   dx/dxi = a1 + a4 eta + a5 zeta + a7 eta zeta,  dx/deta = a2 + a4 xi + a6 zeta + a7 xi zeta,
//   dx/dzeta = a3 + a5 xi + a6 eta + a7 xi eta:
// with one or two reference coordinates fixed per thread every column is affine in the remaining one.
struct TrilinearMonomials
{
  double m[7][3];
  // from the cell's vertices v[k][i], k = 4a + 2b + c
  __device__ __forceinline__ void from_vertices(const double (&v)[8][3])
  {
#pragma unroll
    for (int i = 0; i < 3; ++i)
    {
      m[0][i] = v[4][i] - v[0][i];
      m[1][i] = v[2][i] - v[0][i];
      m[2][i] = v[1][i] - v[0][i];
      m[3][i] = (v[6][i] - v[4][i]) - (v[2][i] - v[0][i]);
      m[4][i] = (v[5][i] - v[4][i]) - (v[1][i] - v[0][i]);
      m[5][i] = (v[3][i] - v[2][i]) - (v[1][i] - v[0][i]);
      m[6][i] = ((v[7][i] - v[6][i]) - (v[5][i] - v[4][i])) - ((v[3][i] - v[2][i]) - (v[1][i] - v[0][i]));
    }
  }
  // the cell with geometry dofs gd (the unit cube when gd is null: finite, inert geometry for idle threads)
  __device__ __forceinline__ void load(const double* __restrict__ xgeom, const int32_t* gd)
  {
    double v[8][3];
#pragma unroll
    for (int k = 0; k < 8; ++k)
    {
      const int32_t d = gd ? gd[k] : 0;
#pragma unroll
      for (int i = 0; i < 3; ++i)
        v[k][i] = gd ? xgeom[3ll * d + i] : (double)((k >> (2 - i)) & 1);
    }
    from_vertices(v);
  }
};

// One thread per (cell position, quadrature point).  J = sum_k x_k dphi_k, K = adj(J),
// G = w K K^T / detJ with 6 unique entries (xx,xy,xz,yy,yz,zz).  Also used for detJ only.
template <bool WRITE_G>
__global__ void k_geometry(int P, const double* __restrict__ xgeom,
                           const int32_t* __restrict__ geom_dofmap,
                           const int32_t* __restrict__ perm, double* __restrict__ G,
                           double* __restrict__ detj_w, int n_list, bool literal_detj, Lay lay)
{
  const int n = P + 1, n2 = n * n, n3 = n2 * n;
  const long long total = (long long)n_list * n3;
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nth)
  {
    const long long p = t / n3;
    const int q = (int)(t - p * n3);
    const int ix = q / n2, iy = (q / n) % n, iz = q % n;
    const double xi[3] = {c_pts[P][ix], c_pts[P][iy], c_pts[P][iz]};
    const int32_t* gd = geom_dofmap + (long long)perm[p] * 8;
    double J[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
#pragma unroll
    for (int k = 0; k < 8; ++k)
    {
      const int a = (k >> 2) & 1, b = (k >> 1) & 1, c = k & 1;
      const double la = a ? xi[0] : 1.0 - xi[0], lb = b ? xi[1] : 1.0 - xi[1],
                   lc = c ? xi[2] : 1.0 - xi[2];
      const double da = a ? 1.0 : -1.0, db = b ? 1.0 : -1.0, dc = c ? 1.0 : -1.0;
      const double dphi[3] = {da * lb * lc, la * db * lc, la * lb * dc};
      const double* xv = xgeom + 3ll * gd[k];
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j)
          J[i][j] += xv[i] * dphi[j];
    }
    double K[3][3];
    K[0][0] = J[1][1] * J[2][2] - J[1][2] * J[2][1];
    K[0][1] = -J[0][1] * J[2][2] + J[0][2] * J[2][1];
    K[0][2] = J[0][1] * J[1][2] - J[0][2] * J[1][1];
    K[1][0] = -J[1][0] * J[2][2] + J[1][2] * J[2][0];
    K[1][1] = J[0][0] * J[2][2] - J[0][2] * J[2][0];
    K[1][2] = -J[0][0] * J[1][2] + J[0][2] * J[1][0];
    K[2][0] = J[1][0] * J[2][1] - J[1][1] * J[2][0];
    K[2][1] = -J[0][0] * J[2][1] + J[0][1] * J[2][0];
    K[2][2] = J[0][0] * J[1][1] - J[0][1] * J[1][0];
    double detJ;
    if (literal_detj) // expression of src/laplacian.hpp:97 (quirk Q17)
      detJ = J[0][0] * K[0][0] - J[1][0] * K[0][1] + J[0][2] * K[2][0];
    else
      detJ = J[0][0] * K[0][0] + J[0][1] * K[1][0] + J[0][2] * K[2][0];
    const double w = c_wts[P][ix] * c_wts[P][iy] * c_wts[P][iz];
    if (WRITE_G)
    {
      const double s = w / detJ;
      G[lay.g_index(p, 0, q)] = (K[0][0] * K[0][0] + K[0][1] * K[0][1] + K[0][2] * K[0][2]) * s;
      G[lay.g_index(p, 1, q)] = (K[1][0] * K[0][0] + K[1][1] * K[0][1] + K[1][2] * K[0][2]) * s;
      G[lay.g_index(p, 2, q)] = (K[2][0] * K[0][0] + K[2][1] * K[0][1] + K[2][2] * K[0][2]) * s;
      G[lay.g_index(p, 3, q)] = (K[1][0] * K[1][0] + K[1][1] * K[1][1] + K[1][2] * K[1][2]) * s;
      G[lay.g_index(p, 4, q)] = (K[2][0] * K[1][0] + K[2][1] * K[1][1] + K[2][2] * K[1][2]) * s;
      G[lay.g_index(p, 5, q)] = (K[2][0] * K[2][0] + K[2][1] * K[2][1] + K[2][2] * K[2][2]) * s;
    }
    else
      detj_w[t] = w * fabs(detJ);
  }
}

// Where the set-up kernels (diagonal, CSR assembly, get_G) read G(p, comp, q) from: the stored array, or
// computed from the vertices on the fly (PMGX_LAP_RECOMPUTE_G: no per-point geometry exists)
struct StoredG
{
  const double* G;
  Lay lay;
  __device__ __forceinline__ double operator()(long long p, int comp, int q) const { return G[lay.g_index(p, comp, q)]; }
};
struct VertexG
{
  const double* xgeom;
  const int32_t* geom_dofmap;
  const int32_t* perm;
  int P;
  bool literal_detj;
  __device__ double operator()(long long p, int comp, int q) const
  {
    const int n = P + 1, ix = q / (n * n), iy = (q / n) % n, iz = q % n;
    const double xi[3] = {c_pts[P][ix], c_pts[P][iy], c_pts[P][iz]};
    double J[3][3], g[6];
    jacobian_at(xgeom, geom_dofmap + (long long)perm[p] * 8, xi, J);
    g_from_jacobian(J, literal_detj, c_wts[P][ix] * c_wts[P][iy] * c_wts[P][iz], g);
    return g[comp];
  }
};

// Per cell: Gc = K K^T / det J of the trilinear map at the cell centre (weight 1), and the affinity
// test: a cell is affine iff every vertex equals v000 + a e1 + b e2 + c e3; the deviation is
// measured against the longest edge.  One thread per launch position.
__global__ void k_cell_geometry(const double* __restrict__ xgeom, const int32_t* __restrict__ geom_dofmap,
                                const int32_t* __restrict__ perm, double* __restrict__ Gc, int n_list,
                                bool literal_detj, double tol, int* __restrict__ n_nonaffine)
{
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_list)
    return;
  const int32_t* gd = geom_dofmap + (long long)perm[p] * 8;
  double v[8][3];
#pragma unroll
  for (int k = 0; k < 8; ++k)
#pragma unroll
    for (int i = 0; i < 3; ++i)
      v[k][i] = xgeom[3ll * gd[k] + i];
  // tensor-product vertex order: k = 4a + 2b + c (src/mesh.hpp:75-84)
  double scale = 0.0, dev = 0.0;
#pragma unroll
  for (int i = 0; i < 3; ++i)
  {
    const double e1 = v[4][i] - v[0][i], e2 = v[2][i] - v[0][i], e3 = v[1][i] - v[0][i];
    scale = fmax(scale, fmax(fabs(e1), fmax(fabs(e2), fabs(e3))));
    dev = fmax(dev, fabs(v[6][i] - (v[0][i] + e1 + e2)));
    dev = fmax(dev, fabs(v[5][i] - (v[0][i] + e1 + e3)));
    dev = fmax(dev, fabs(v[3][i] - (v[0][i] + e2 + e3)));
    dev = fmax(dev, fabs(v[7][i] - (v[0][i] + e1 + e2 + e3)));
  }
  if (!(dev <= tol * scale))
    atomicAdd(n_nonaffine, 1);
  double J[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
#pragma unroll
  for (int k = 0; k < 8; ++k)
  {
    const int a = (k >> 2) & 1, b = (k >> 1) & 1, c = k & 1;
    const double dphi[3] = {(a ? 1.0 : -1.0) * 0.25, (b ? 1.0 : -1.0) * 0.25, (c ? 1.0 : -1.0) * 0.25};
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j)
        J[i][j] += v[k][i] * dphi[j];
  }
  double K[3][3];
  K[0][0] = J[1][1] * J[2][2] - J[1][2] * J[2][1];
  K[0][1] = -J[0][1] * J[2][2] + J[0][2] * J[2][1];
  K[0][2] = J[0][1] * J[1][2] - J[0][2] * J[1][1];
  K[1][0] = -J[1][0] * J[2][2] + J[1][2] * J[2][0];
  K[1][1] = J[0][0] * J[2][2] - J[0][2] * J[2][0];
  K[1][2] = -J[0][0] * J[1][2] + J[0][2] * J[1][0];
  K[2][0] = J[1][0] * J[2][1] - J[1][1] * J[2][0];
  K[2][1] = -J[0][0] * J[2][1] + J[0][1] * J[2][0];
  K[2][2] = J[0][0] * J[1][1] - J[0][1] * J[1][0];
  const double detJ = literal_detj ? J[0][0] * K[0][0] - J[1][0] * K[0][1] + J[0][2] * K[2][0]
                                   : J[0][0] * K[0][0] + J[0][1] * K[1][0] + J[0][2] * K[2][0];
  const double s = 1.0 / detJ;
  double* g = Gc + (size_t)p * 6;
  g[0] = (K[0][0] * K[0][0] + K[0][1] * K[0][1] + K[0][2] * K[0][2]) * s;
  g[1] = (K[1][0] * K[0][0] + K[1][1] * K[0][1] + K[1][2] * K[0][2]) * s;
  g[2] = (K[2][0] * K[0][0] + K[2][1] * K[0][1] + K[2][2] * K[0][2]) * s;
  g[3] = (K[1][0] * K[1][0] + K[1][1] * K[1][1] + K[1][2] * K[1][2]) * s;
  g[4] = (K[2][0] * K[1][0] + K[2][1] * K[1][1] + K[2][2] * K[1][2]) * s;
  g[5] = (K[2][0] * K[2][0] + K[2][1] * K[2][1] + K[2][2] * K[2][2]) * s;
}

// ------------------------------------------------------ geometry of the 27-node hexahedron --
// PMGX_LAP_GEOM_Q2: the triquadratic map x(xi) = sum_k x_k L_a(xi) L_b(eta) L_c(zeta) with node k = 9a + 3b + c at
// reference coordinates {0, 1/2, 1}^3.  The corners are k = 18a' + 6b' + 2c' for the trilinear vertex (a',b',c').
constexpr int Q2_NODES = 27;

// the quadratic Lagrange basis on {0, 1/2, 1} and its derivative at t
__device__ __forceinline__ void q2_basis(double t, double (&l)[3], double (&d)[3])
{
  l[0] = (2.0 * t - 1.0) * (t - 1.0);
  l[1] = 4.0 * t * (1.0 - t);
  l[2] = t * (2.0 * t - 1.0);
  d[0] = 4.0 * t - 3.0;
  d[1] = 4.0 - 8.0 * t;
  d[2] = 4.0 * t - 1.0;
}

// J at xi of the cell whose node coordinates are X(k, i), by sum factorisation over the 3 x 3 x 3 basis: the zeta
// direction first (value and derivative), then eta, then xi.
template <typename Nodes>
__device__ __forceinline__ void jacobian_q2(const Nodes& X, const double (&xi)[3], double (&J)[3][3])
{
  double la[3], da[3], lb[3], db[3], lc[3], dc[3];
  q2_basis(xi[0], la, da);
  q2_basis(xi[1], lb, db);
  q2_basis(xi[2], lc, dc);
#pragma unroll
  for (int i = 0; i < 3; ++i)
  {
    double j0 = 0.0, j1 = 0.0, j2 = 0.0;
#pragma unroll
    for (int a = 0; a < 3; ++a)
    {
      double u = 0.0, ueta = 0.0, uzeta = 0.0; // sum_bc x L_b L_c, x L_b' L_c, x L_b L_c'
#pragma unroll
      for (int b = 0; b < 3; ++b)
      {
        double s = 0.0, t = 0.0; // sum_c x L_c, x L_c'
#pragma unroll
        for (int c = 0; c < 3; ++c)
        {
          const double x = X(9 * a + 3 * b + c, i);
          s = fma(x, lc[c], s);
          t = fma(x, dc[c], t);
        }
        u = fma(s, lb[b], u);
        ueta = fma(s, db[b], ueta);
        uzeta = fma(t, lb[b], uzeta);
      }
      j0 = fma(u, da[a], j0);
      j1 = fma(ueta, la[a], j1);
      j2 = fma(uzeta, la[a], j2);
    }
    J[i][0] = j0, J[i][1] = j1, J[i][2] = j2;
  }
}

// G (WRITE_G) or w |det J| at every quadrature point of the 27-node cells.  One warp per launch position: the warp
// stages the cell's 27 x 3 coordinates in shared memory once, then each lane forms J at its points from the staged
// copy and G = w K K^T / det J through the same helpers as every other path.
constexpr int Q2_GEOM_WARPS = 8;
template <bool WRITE_G>
__global__ void __launch_bounds__(32 * Q2_GEOM_WARPS)
    k_geometry_q2(int P, const double* __restrict__ xgeom, const int32_t* __restrict__ geom_dofmap,
                  const int32_t* __restrict__ perm, double* __restrict__ G, double* __restrict__ detj_w, int n_list,
                  bool literal_detj, Lay lay)
{
  __shared__ double nodes[Q2_GEOM_WARPS][Q2_NODES * 3];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* xs = nodes[warp];
  const auto X = [xs](int k, int i) { return xs[3 * k + i]; };
  const int n = P + 1, n2 = n * n, n3 = n2 * n;
  const long long stride = (long long)gridDim.x * Q2_GEOM_WARPS;
  for (long long p = (long long)blockIdx.x * Q2_GEOM_WARPS + warp; p < n_list; p += stride)
  {
    const int32_t* gd = geom_dofmap + (long long)perm[p] * Q2_NODES;
    for (int e = lane; e < Q2_NODES * 3; e += 32)
      xs[e] = xgeom[3ll * gd[e / 3] + e % 3];
    __syncwarp();
    for (int q = lane; q < n3; q += 32)
    {
      const int ix = q / n2, iy = (q / n) % n, iz = q % n;
      const double xi[3] = {c_pts[P][ix], c_pts[P][iy], c_pts[P][iz]};
      const double w = c_wts[P][ix] * c_wts[P][iy] * c_wts[P][iz];
      double J[3][3], K[3][3];
      jacobian_q2(X, xi, J);
      const double detJ = adjugate_det(J, literal_detj, K);
      if (WRITE_G)
      {
        double g[6];
        g_from_adjugate(K, w / detJ, g);
#pragma unroll
        for (int c = 0; c < 6; ++c)
          G[lay.g_index(p, c, q)] = g[c];
      }
      else
        detj_w[p * n3 + q] = w * fabs(detJ);
    }
    __syncwarp(); // the next cell overwrites xs
  }
}

// Per cell: Gc = K K^T / det J of the triquadratic map at the cell centre (weight 1), and the affinity test: a cell is
// affine iff every node equals v000 + (a/2) e1 + (b/2) e2 + (c/2) e3 (e1, e2, e3 the edges from v000), measured
// against the longest edge like k_cell_geometry.  One thread per launch position.
__global__ void k_cell_geometry_q2(const double* __restrict__ xgeom, const int32_t* __restrict__ geom_dofmap,
                                   const int32_t* __restrict__ perm, double* __restrict__ Gc, int n_list,
                                   bool literal_detj, double tol, int* __restrict__ n_nonaffine)
{
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_list)
    return;
  const int32_t* gd = geom_dofmap + (long long)perm[p] * Q2_NODES;
  const auto X = [xgeom, gd](int k, int i) { return xgeom[3ll * gd[k] + i]; };
  double scale = 0.0, dev = 0.0;
#pragma unroll
  for (int i = 0; i < 3; ++i)
  {
    const double v0 = X(0, i), e1 = X(18, i) - v0, e2 = X(6, i) - v0, e3 = X(2, i) - v0;
    scale = fmax(scale, fmax(fabs(e1), fmax(fabs(e2), fabs(e3))));
    for (int k = 1; k < Q2_NODES; ++k)
    {
      const int a = k / 9, b = (k / 3) % 3, c = k % 3;
      dev = fmax(dev, fabs(X(k, i) - (v0 + 0.5 * (a * e1 + b * e2 + c * e3))));
    }
  }
  if (!(dev <= tol * scale))
    atomicAdd(n_nonaffine, 1);
  const double centre[3] = {0.5, 0.5, 0.5};
  double J[3][3], K[3][3], g[6];
  jacobian_q2(X, centre, J);
  const double detJ = adjugate_det(J, literal_detj, K);
  g_from_adjugate(K, 1.0 / detJ, g);
#pragma unroll
  for (int c = 0; c < 6; ++c)
    Gc[(size_t)p * 6 + c] = g[c];
}

// Per-thread factored Jacobians of the apply kernels that recompute G.  Along a line of fixed (eta, zeta) (a
// column thread, an mma lane): dx/dxi is constant, dx/deta and dx/dzeta are affine in xi -- 15 coefficients, 6 FMAs
// per point.
struct JacobianAlongXi
{
  double c0[3], e0[3], e1[3], z0[3], z1[3];
  __device__ __forceinline__ void init(const TrilinearMonomials& M, double eta, double zeta)
  {
#pragma unroll
    for (int i = 0; i < 3; ++i)
    {
      c0[i] = fma(M.m[6][i] * eta + M.m[4][i], zeta, fma(M.m[3][i], eta, M.m[0][i]));
      e0[i] = fma(M.m[5][i], zeta, M.m[1][i]);
      e1[i] = fma(M.m[6][i], zeta, M.m[3][i]);
      z0[i] = fma(M.m[5][i], eta, M.m[2][i]);
      z1[i] = fma(M.m[6][i], eta, M.m[4][i]);
    }
  }
  __device__ __forceinline__ void at(double xi, double (&J)[3][3]) const
  {
#pragma unroll
    for (int i = 0; i < 3; ++i)
    {
      J[i][0] = c0[i];
      J[i][1] = fma(e1[i], xi, e0[i]);
      J[i][2] = fma(z1[i], xi, z0[i]);
    }
  }
};
// On a plane of fixed zeta (a slab thread): dx/dxi = x0 + x1 eta, dx/deta = y0 + x1 xi and
// dx/dzeta = (a3 + a5 xi) + (a6 + a7 xi) eta -- 21 coefficients, kept in shared memory (store); per plane xi
// 9 FMAs (plane), per point 6 (at).
struct JacobianAtZeta
{
  double x0[3], x1[3], y0[3], a3[3], a5[3], a6[3], a7[3];
  __device__ __forceinline__ void init(const TrilinearMonomials& M, double zeta)
  {
#pragma unroll
    for (int i = 0; i < 3; ++i)
    {
      x0[i] = fma(M.m[4][i], zeta, M.m[0][i]);
      x1[i] = fma(M.m[6][i], zeta, M.m[3][i]);
      y0[i] = fma(M.m[5][i], zeta, M.m[1][i]);
      a3[i] = M.m[2][i], a5[i] = M.m[4][i], a6[i] = M.m[5][i], a7[i] = M.m[6][i];
    }
  }
  // the 21 coefficients as rows of a [21][stride] array
  __device__ __forceinline__ void store(double* p, int stride) const
  {
#pragma unroll
    for (int i = 0; i < 3; ++i)
    {
      p[(0 + i) * stride] = x0[i], p[(3 + i) * stride] = x1[i], p[(6 + i) * stride] = y0[i];
      p[(9 + i) * stride] = a3[i], p[(12 + i) * stride] = a5[i], p[(15 + i) * stride] = a6[i];
      p[(18 + i) * stride] = a7[i];
    }
  }
  // the xi-dependent parts of plane xi: dx/deta, and dx/dzeta = z0 + z1 eta
  struct Plane
  {
    double y[3], z0[3], z1[3];
  };
  // plane() and at() on the stored form, reading each coefficient where it is used (no 21 live registers)
  __device__ __forceinline__ static Plane plane(const volatile double* p, int stride, double xi)
  {
    Plane q;
#pragma unroll
    for (int i = 0; i < 3; ++i)
    {
      q.y[i] = fma(p[(3 + i) * stride], xi, p[(6 + i) * stride]);
      q.z0[i] = fma(p[(12 + i) * stride], xi, p[(9 + i) * stride]);
      q.z1[i] = fma(p[(18 + i) * stride], xi, p[(15 + i) * stride]);
    }
    return q;
  }
  __device__ __forceinline__ static void at(const volatile double* p, int stride, const Plane& q, double eta,
                                            double (&J)[3][3])
  {
#pragma unroll
    for (int i = 0; i < 3; ++i)
    {
      J[i][0] = fma(p[(3 + i) * stride], eta, p[(0 + i) * stride]);
      J[i][1] = q.y[i];
      J[i][2] = fma(q.z1[i], eta, q.z0[i]);
    }
  }
};

// diag(A) contributions, thread per (cell position, local dof); see DESIGN.md "diagonal".
template <typename Geo>
__global__ void k_diag(int P, Geo G, const int32_t* __restrict__ enc,
                       const int32_t* __restrict__ perm, const double* __restrict__ kappa,
                       double* __restrict__ diag, int n_list, Lay lay)
{
  const int n = P + 1, n2 = n * n, n3 = n2 * n;
  const long long total = (long long)n_list * n3;
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nth)
  {
    const long long p = t / n3;
    const int a = (int)(t - p * n3);
    const int32_t d = enc[lay.enc_index(p, a)];
    if (d < 0)
      continue;
    const int i = a / n2, j = (a / n) % n, k = a % n;
    const double* D = c_D[P];
    double s = 0.0;
    for (int q = 0; q < n; ++q)
    {
      const double dx = D[q * n + i], dy = D[q * n + j], dz = D[q * n + k];
      s += dx * dx * G(p, 0, q * n2 + j * n + k);
      s += dy * dy * G(p, 3, i * n2 + q * n + k);
      s += dz * dz * G(p, 5, i * n2 + j * n + q);
    }
    const double dii = D[i * n + i], djj = D[j * n + j], dkk = D[k * n + k];
    s += 2.0 * (G(p, 1, a) * dii * djj + G(p, 2, a) * dii * dkk
                + G(p, 4, a) * djj * dkk);
    atomicAdd(&diag[d], kappa[perm[p]] * s);
  }
}

__global__ void k_invert_diag(const double* __restrict__ diag, const int8_t* __restrict__ bc,
                              double* __restrict__ dinv, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
    dinv[i] = bc[i] ? 1.0 : 1.0 / diag[i];
}

template <typename Geo>
__global__ void k_G_to_reference_layout(Geo G, double* __restrict__ out, int n3, long long total)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nth)
  {
    const long long p = t / (6 * n3);
    const int r = (int)(t - p * 6 * n3);
    const int q = r / 6, c = r % 6;
    out[t] = G(p, c, q);
  }
}

__global__ void k_rhs(const double* __restrict__ detj_w, const int32_t* __restrict__ enc,
                      const double* __restrict__ fvals, double* __restrict__ b, long long total,
                      int n3, Lay lay)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nth)
  {
    const int32_t d = enc[lay.enc_index(t / n3, (int)(t % n3))];
    if (d >= 0)
      atomicAdd(&b[d], fvals[d] * detj_w[t]);
  }
}

__global__ void k_set_bc_value(double* __restrict__ b, const int8_t* __restrict__ bc, double g, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && bc[i])
    b[i] = g;
}

// gbc = bc ? g : 0
__global__ void k_mask_to_bc(const double* __restrict__ g, const int8_t* __restrict__ bc, double* __restrict__ gbc, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
    gbc[i] = bc[i] ? g[i] : 0.0;
}

// b = bc ? g : b - y   (lifting on the free rows, set_bc on the marked ones)
__global__ void k_lift(double* __restrict__ b, const double* __restrict__ y, const double* __restrict__ g,
                       const int8_t* __restrict__ bc, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
    b[i] = bc[i] ? g[i] : y[i] * (-1.0) + b[i];
}

__global__ void k_fill(double* __restrict__ v, double a, int n)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
    v[i] = a;
}

// ------------------------------------------------------------- CSR assembly kernels --
// Entry (i,j) of the element matrix kappa * B^T G B with the collocated gradient table
// (phi = identity at the GLL points, src/laplacian.hpp:200-202): only index pairs that
// agree in at least one direction couple.
template <typename Geo>
__device__ double element_entry(int P, const Geo& G, long long p, int i, int j)
{
  const int n = P + 1, n2 = n * n;
  const double* D = c_D[P];
  const int ix = i / n2, iy = (i / n) % n, iz = i % n;
  const int jx = j / n2, jy = (j / n) % n, jz = j % n;
  double s = 0.0;
  if (iy == jy && iz == jz)
    for (int q = 0; q < n; ++q)
      s += D[q * n + ix] * D[q * n + jx] * G(p, 0, q * n2 + iy * n + iz);
  if (ix == jx && iz == jz)
    for (int q = 0; q < n; ++q)
      s += D[q * n + iy] * D[q * n + jy] * G(p, 3, ix * n2 + q * n + iz);
  if (ix == jx && iy == jy)
    for (int q = 0; q < n; ++q)
      s += D[q * n + iz] * D[q * n + jz] * G(p, 5, ix * n2 + iy * n + q);
  if (iz == jz)
    s += D[jx * n + ix] * D[iy * n + jy] * G(p, 1, jx * n2 + iy * n + iz)
         + D[jy * n + iy] * D[ix * n + jx] * G(p, 1, ix * n2 + jy * n + iz);
  if (iy == jy)
    s += D[jx * n + ix] * D[iz * n + jz] * G(p, 2, jx * n2 + iy * n + iz)
         + D[jz * n + iz] * D[ix * n + jx] * G(p, 2, ix * n2 + iy * n + jz);
  if (ix == jx)
    s += D[jy * n + iy] * D[iz * n + jz] * G(p, 4, ix * n2 + jy * n + iz)
         + D[jz * n + iz] * D[iy * n + jy] * G(p, 4, ix * n2 + iy * n + jz);
  return s;
}

// One (key, value) per (cell, i, j); key = row * ntot + col, sentinel for dropped entries
// (ghost rows, Dirichlet rows / columns: fem::assemble_matrix with bcs, src/csr.hpp:84).
template <typename Geo>
__global__ void k_element_triplets(int P, Geo G, const int32_t* __restrict__ enc,
                                   const int32_t* __restrict__ perm, const double* __restrict__ kappa,
                                   long long n_list, int n_owned, long long ntot,
                                   unsigned long long* __restrict__ keys, double* __restrict__ vals, Lay lay)
{
  const int n = P + 1, n3 = n * n * n;
  const long long per_cell = (long long)n3 * n3;
  const long long total = n_list * per_cell;
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nth)
  {
    const long long p = t / per_cell;
    const int r = (int)(t - p * per_cell);
    const int i = r / n3, j = r - i * n3;
    const int32_t di = enc[lay.enc_index(p, i)], dj = enc[lay.enc_index(p, j)];
    if (di < 0 || dj < 0 || di >= n_owned)
    {
      keys[t] = ~0ull;
      vals[t] = 0.0;
      continue;
    }
    keys[t] = (unsigned long long)di * (unsigned long long)ntot + (unsigned long long)dj;
    vals[t] = kappa[perm[p]] * element_entry(P, G, p, i, j);
  }
}

// Dirichlet rows: unit diagonal (fem::set_diagonal, src/csr.hpp:86)
__global__ void k_bc_diag_triplets(const int8_t* __restrict__ bc, int n_owned, long long ntot,
                                   unsigned long long* __restrict__ keys, double* __restrict__ vals)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_owned)
    return;
  keys[i] = bc[i] ? (unsigned long long)i * (unsigned long long)ntot + (unsigned long long)i : ~0ull;
  vals[i] = bc[i] ? 1.0 : 0.0;
}

__global__ void k_split_keys(const unsigned long long* __restrict__ keys, long long nnz, long long ntot,
                             int n_owned, int32_t* __restrict__ cols, int32_t* __restrict__ row_count,
                             int32_t* __restrict__ owned_count)
{
  const long long nth = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < nnz; t += nth)
  {
    const unsigned long long k = keys[t];
    const int row = (int)(k / (unsigned long long)ntot);
    const int col = (int)(k - (unsigned long long)row * (unsigned long long)ntot);
    cols[t] = col;
    atomicAdd(&row_count[row], 1);
    if (col < n_owned)
      atomicAdd(&owned_count[row], 1);
  }
}

__global__ void k_offdiag(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ owned_count,
                          int n_rows, int32_t* __restrict__ off_diag)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_rows)
    off_diag[i] = row_ptr[i] + owned_count[i];
}

// ---------------------------------------------------------------- apply launches --
// One launch of an apply kernel: the cells [cell0, cell0 + count) of the launch list, whose first
// batch in the SLAB layout is batch0 (the COLUMN-layout kernels ignore it); geom is Gc for the
// kernels that take one geometry 6-vector per cell, G for the streamed-G kernels.  The kernels that
// recompute G per point read the mesh instead: xgeom, geom_dofmap (both borrowed) and the det J form.
struct ApplyArgs
{
  const double* x;
  double* y;
  const double* geom;
  const int32_t* enc;
  const int32_t* perm;
  const double* kappa;
  long long batch0;
  int cell0, count;
  const double* xgeom;
  const int32_t* geom_dofmap;
  int literal_detj;
};

// Launches a persistent apply kernel of degree P: CTAs of tpb threads stay resident and walk over the
// n_blocks blocks of work (blockIdx.x, + gridDim.x, ...), so exactly as many are launched as fit on the
// device at once.  The shared-memory opt-in and the occupancy query run once per device and kernel.
template <auto kernel, typename... Tail>
void launch_persistent(pmgx_ctx* c, cudaStream_t st, const ApplyArgs& a, const char* name, int P, int tpb,
                       size_t smem, int n_blocks, Tail... tail)
{
  if (a.count <= 0)
    return;
  static int ctas_per_sm[64] = {0};
  if (ctas_per_sm[c->device] == 0)
  {
    PMGX_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int nb = 0;
    PMGX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, tpb, smem));
    PMGX_REQUIRE(nb >= 1, "%s (P%d) does not fit on an SM", name, P);
    ctas_per_sm[c->device] = nb;
  }
  const int grid = std::min(n_blocks, ctas_per_sm[c->device] * c->num_sms);
  const bool timed = c->profiling && a.cell0 == 0; // per-kernel timing covers the interior-cell launch only
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (timed)
  {
    PMGX_CUDA(cudaEventCreate(&e0));
    PMGX_CUDA(cudaEventCreate(&e1));
    PMGX_CUDA(cudaEventRecord(e0, st));
  }
  kernel<<<grid, tpb, smem, st>>>(a.x, a.y, a.geom, a.enc, a.perm, a.kappa, tail...);
  check_launch(name);
  count_launch(c);
  if (timed)
  {
    PMGX_CUDA(cudaEventRecord(e1, st));
    c->prof[P].emplace_back(e0, e1);
  }
}

// The SLAB-layout kernels (k_apply_tma, k_apply_affine*): one block of work is one batch of Cfg::cpb cells
template <auto kernel, typename Cfg, typename... Extra>
void launch_batched(pmgx_ctx* c, cudaStream_t st, const ApplyArgs& a, const char* name, Extra... extra)
{
  const int nbatch = (a.count + Cfg::cpb - 1) / Cfg::cpb;
  launch_persistent<kernel>(c, st, a, name, Cfg::n - 1, Cfg::tpb, Cfg::smem, nbatch, a.batch0, a.cell0, a.count,
                            nbatch, extra...);
}

// Every launcher below (one per kernel family) exports
//   cell_geometry  the kernel reads Gc (one geometry 6-vector per affine cell) instead of G
//   cpb            cells per batch of the SLAB layout; 0: the kernel reads the COLUMN layout
//   name()         the kernel and its template arguments, as pmgx_laplacian_kernel_name reports them
//   launch()

// ------------------------------------------------------------ the column apply kernel --
// smem row stride: pad when a (j -> j+1) step of n doubles would alias banks (n % 8 == 0)
template <int P>
struct ApplyCfg
{
  static constexpr int n = P + 1;
  static constexpr int n2 = n * n;
  static constexpr int n3 = n2 * n;
  static constexpr int row = (n % 8 == 0) ? n + 1 : n;
  static constexpr int plane = n * row;
  // threads per block: the smallest of {128,192,256} wasting the fewest lanes
  static constexpr int tpb = P == 8 ? 256 : 128;
  static constexpr int cpb = tpb / n2; // cells per block
  static constexpr int smem_doubles = cpb * (n * plane + 4 * plane);
};

// RECOMPUTE: no G array; the thread forms G at its (j, k) column's point of every plane i from the cell's vertices
template <int P, bool RECOMPUTE>
__global__ void __launch_bounds__(ApplyCfg<P>::tpb)
k_apply(const double* __restrict__ x, double* __restrict__ y, const double* __restrict__ G,
        const int32_t* __restrict__ enc, const int32_t* __restrict__ perm,
        const double* __restrict__ kappa, int first, int count, const double* __restrict__ xgeom,
        const int32_t* __restrict__ geom_dofmap, int literal_detj)
{
  using C = ApplyCfg<P>;
  constexpr int n = C::n, n2 = C::n2, n3 = C::n3, ROW = C::row, PL = C::plane, CPB = C::cpb;
  extern __shared__ double smem[];
  double* su = smem;                      // [CPB][n][PL]
  double* sf = smem + CPB * n * PL;       // [2][CPB][2][PL]

  const int tid = threadIdx.x;
  const int cl = tid / n2;
  const int jk = tid - cl * n2;
  const int j = jk / n, k = jk - j * n;
  const long long pl = (long long)blockIdx.x * CPB + cl;
  const bool active = (cl < CPB) && (pl < count);
  const long long p = first + pl;
  const int sjk = j * ROW + k;

  int d[n];
  double u[n];
  double kap = 0.0;
  const double* Gp = G + p * 6 * n3 + jk;
  double g[6];
  JacobianAlongXi jac;   // RECOMPUTE
  double wjk = 0.0;      // RECOMPUTE: w_j w_k
  if constexpr (RECOMPUTE)
  {
    TrilinearMonomials M;
    M.load(xgeom, active ? geom_dofmap + (long long)perm[p] * 8 : nullptr);
    jac.init(M, c_pts[P][j], c_pts[P][k]);
    wjk = c_wts[P][j] * c_wts[P][k];
  }
  if (active)
  {
    const int32_t* e = enc + p * n3 + jk;
#pragma unroll
    for (int i = 0; i < n; ++i)
      d[i] = ldg_stream_i32(e + i * n2);
    if constexpr (!RECOMPUTE)
    {
#pragma unroll
      for (int c = 0; c < 6; ++c)
        g[c] = ldg_stream(Gp + c * n3);
    }
    kap = kappa[perm[p]];
#pragma unroll
    for (int i = 0; i < n; ++i)
    {
      const int idx = d[i] < 0 ? ~d[i] : d[i];
      const double xv = x[idx];
      if (d[i] < 0)
        y[idx] = xv; // Dirichlet row: y = x (src/laplacian.hpp:273-274)
      u[i] = d[i] < 0 ? 0.0 : xv;
      su[(cl * n + i) * PL + sjk] = u[i];
    }
  }
  else
  {
#pragma unroll
    for (int i = 0; i < n; ++i)
      u[i] = 0.0, d[i] = -1;
#pragma unroll
    for (int c = 0; c < 6; ++c)
      g[c] = 0.0;
  }
  // rows of D needed with a runtime index
  double Dj[n], Dk[n], DTj[n], DTk[n];
#pragma unroll
  for (int l = 0; l < n; ++l)
  {
    Dj[l] = c_D[P][j * n + l];
    Dk[l] = c_D[P][k * n + l];
    DTj[l] = c_D[P][l * n + j];
    DTk[l] = c_D[P][l * n + k];
  }
  double acc[n];
#pragma unroll
  for (int i = 0; i < n; ++i)
    acc[i] = 0.0;
  __syncthreads();

  const int cls = active ? cl : 0;
#pragma unroll
  for (int i = 0; i < n; ++i)
  {
    // prefetch next plane's geometry
    double gn[6];
    if constexpr (RECOMPUTE)
    {
      double J[3][3];
      jac.at(c_pts[P][i], J);
      g_from_jacobian(J, literal_detj, c_wts[P][i] * wjk, g);
    }
    else if (i + 1 < n)
    {
      if (active)
      {
#pragma unroll
        for (int c = 0; c < 6; ++c)
          gn[c] = ldg_stream(Gp + c * n3 + (i + 1) * n2);
      }
      else
      {
#pragma unroll
        for (int c = 0; c < 6; ++c)
          gn[c] = 0.0;
      }
    }
    // gradient at quadrature point (i, j, k)
    double gx = 0.0, gy = 0.0, gz = 0.0;
    const double* sp = su + (cls * n + i) * PL;
#pragma unroll
    for (int l = 0; l < n; ++l)
    {
      gx = fma(c_D[P][i * n + l], u[l], gx);
      gy = fma(Dj[l], sp[l * ROW + k], gy);
      gz = fma(Dk[l], sp[j * ROW + l], gz);
    }
    const double fx = kap * (g[0] * gx + g[1] * gy + g[2] * gz);
    const double fy = kap * (g[1] * gx + g[3] * gy + g[4] * gz);
    const double fz = kap * (g[2] * gx + g[4] * gy + g[5] * gz);
#pragma unroll
    for (int l = 0; l < n; ++l)
      acc[l] = fma(c_D[P][i * n + l], fx, acc[l]);
    double* sfy = sf + (((i & 1) * CPB + cls) * 2 + 0) * PL;
    double* sfz = sfy + PL;
    if (active)
    {
      sfy[sjk] = fy;
      sfz[sjk] = fz;
    }
    __syncthreads();
    double t = 0.0;
#pragma unroll
    for (int q = 0; q < n; ++q)
    {
      t = fma(DTj[q], sfy[q * ROW + k], t);
      t = fma(DTk[q], sfz[j * ROW + q], t);
    }
    acc[i] += t;
    if (!RECOMPUTE && i + 1 < n)
    {
#pragma unroll
      for (int c = 0; c < 6; ++c)
        g[c] = gn[c];
    }
  }
  if (active)
  {
#pragma unroll
    for (int i = 0; i < n; ++i)
      if (d[i] >= 0)
        atomicAdd(&y[d[i]], acc[i]);
  }
}

// Not persistent: one CTA per ApplyCfg<P>::cpb cells of the COLUMN layout
template <int P, bool RECOMPUTE = false>
struct ColumnApply
{
  using C = ApplyCfg<P>;
  static constexpr bool cell_geometry = false;
  static constexpr int cpb = 0;
  static void name(char* s, int cap)
  {
    if (RECOMPUTE)
      snprintf(s, cap, "k_apply<%d,recomputed>", P);
    else
      snprintf(s, cap, "k_apply<%d>", P);
  }
  static void launch(pmgx_ctx* c, cudaStream_t st, const ApplyArgs& a)
  {
    if (a.count <= 0)
      return;
    const size_t smem = (size_t)C::smem_doubles * sizeof(double);
    static bool configured[64] = {false};
    if (!configured[c->device])
    {
      PMGX_CUDA(cudaFuncSetAttribute(k_apply<P, RECOMPUTE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      configured[c->device] = true;
    }
    const int grid = (a.count + C::cpb - 1) / C::cpb;
    const bool timed = c->profiling && a.cell0 == 0; // per-kernel timing covers the interior-cell launch only
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (timed)
    {
      PMGX_CUDA(cudaEventCreate(&e0));
      PMGX_CUDA(cudaEventCreate(&e1));
      PMGX_CUDA(cudaEventRecord(e0, st));
    }
    k_apply<P, RECOMPUTE><<<grid, C::tpb, smem, st>>>(a.x, a.y, a.geom, a.enc, a.perm, a.kappa, a.cell0, a.count,
                                                      a.xgeom, a.geom_dofmap, a.literal_detj);
    check_launch("k_apply");
    count_launch(c);
    if (timed)
    {
      PMGX_CUDA(cudaEventRecord(e1, st));
      c->prof[P].emplace_back(e0, e1);
    }
  }
};

// --------------------------------------------- the TMA-pipelined slab apply kernel --
// Thread = one z-index k of one cell; it keeps the whole (ix,iy) slab of the element in
// registers, so the x and y contractions are pure register FMAs with compile-time D entries
// and only the z contraction exchanges data through shared memory (rows of n values that all
// n threads of a cell read as a broadcast).  This moves ~1/3 of the bytes of the column
// kernel through the LSU/shared-memory pipe, which ncu showed to be the limiter there
// (l1tex data-pipe 80 % busy at 61 % DRAM, profiles/r1_apply_p4_column.txt).
// The one-shot streams (geometry factors, encoded dofmap) do not pass through registers with
// the latency exposed to a handful of resident warps: a persistent CTA walks over its batches
// and an elected thread
// keeps a ring of R geometry planes (and the next batch's dofmap) in flight with
// cp.async.bulk (TMA) into shared memory, completion tracked by mbarriers.  Memory-level
// parallelism is then set by the ring depth, not by occupancy or register count.
__device__ __forceinline__ uint32_t smem_u32(const void* p)
{
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init()
{
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
  asm volatile("{\n"
               ".reg .pred p;\n"
               "WAIT_LOOP:\n"
               "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
               "@p bra WAIT_DONE;\n"
               "bra WAIT_LOOP;\n"
               "WAIT_DONE:\n"
               "}\n" ::"r"(smem_u32(bar)),
               "r"(parity)
               : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first()
{
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t pol)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
               "[%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(pol)
               : "memory");
}

// RECOMPUTE: no geometry ring; every thread forms G at its points from the cell's vertices (JacobianAtZeta)
template <int P, int TPB, bool RECOMPUTE = false>
struct TmaCfg
{
  static constexpr int n = P + 1;
  static constexpr int n2 = n * n;
  static constexpr int tpb = TPB;
  static constexpr int R = 2; // geometry planes in flight (measured on B200: a 2-plane ring wins for P3/P4)
  static constexpr int ring = RECOMPUTE ? 0 : R;
  static constexpr int cpb = tpb / n;
  static constexpr int S = (cpb * n + 1) & ~1;  // G rows: 16-byte multiples, (almost) no padding streamed
  static constexpr int SE = (cpb * n + 3) & ~3; // dofmap rows: 16-byte multiples of int32
  static constexpr int minb = P == 1 ? 4 : (P == 2 ? 3 : (TPB <= 64 ? 4 : 2)); // resident CTAs per SM
  static constexpr int kp = n + (n & 1);
  // per-cell stride of a z-row plane buffer: an odd number of 16-byte chunks, so the cells of
  // a warp start in different bank groups (profiles/r1_apply_p3_slab.txt: 75 % of the shared
  // wavefronts were conflict replays with the unpadded stride)
  static constexpr int cs = ((n * kp / 2) & 1) ? n * kp : n * kp + 2;
  static constexpr int plane_doubles = n * 6 * S;
  static constexpr uint32_t plane_bytes = plane_doubles * sizeof(double);
  static constexpr uint32_t enc_bytes = n2 * SE * sizeof(int32_t);
  static constexpr int buf_doubles = 2 * cpb * cs; // double-buffered plane rows (su and sf each)
  // RECOMPUTE: instead of the ring, [21][TPB] JacobianAtZeta coefficients and [n][6][TPB] G at the thread's points
  // of the current plane, one column per thread (written and read by the same thread: no barrier)
  static constexpr int GS = RECOMPUTE ? TPB : S; // stride of the six G components in shared memory
  static constexpr size_t off_gq = 21 * (size_t)TPB * sizeof(double);
  static constexpr size_t off_enc = RECOMPUTE ? off_gq + (size_t)6 * n * TPB * sizeof(double) : (size_t)ring * plane_bytes;
  // dofmap buffers: double-buffered (read again at scatter time, next batch prefetched meanwhile)
  static constexpr size_t off_su = off_enc + 2 * enc_bytes;
  static constexpr size_t off_sf = off_su + (size_t)buf_doubles * sizeof(double);
  static constexpr size_t off_bar = off_sf + (size_t)buf_doubles * sizeof(double);
  static constexpr size_t smem = off_bar + (R + 2) * sizeof(uint64_t);
};

template <int P, int TPB, bool RECOMPUTE>
__global__ void __launch_bounds__(TPB, TmaCfg<P, TPB, RECOMPUTE>::minb)
k_apply_tma(const double* __restrict__ x, double* __restrict__ y, const double* __restrict__ G,
            const int32_t* __restrict__ enc, const int32_t* __restrict__ perm,
            const double* __restrict__ kappa, long long batch0, int cell0, int count, int nbatch,
            const double* __restrict__ xgeom, const int32_t* __restrict__ geom_dofmap, int literal_detj)
{
  using C = TmaCfg<P, TPB, RECOMPUTE>;
  constexpr int n = C::n, n2 = C::n2, CPB = C::cpb, S = C::S, SE = C::SE, KP = C::kp, CS = C::cs, R = C::R;
  constexpr int GS = C::GS;
  extern __shared__ __align__(128) unsigned char smraw[];
  double* sG = reinterpret_cast<double*>(smraw);
  double* const sJ = sG + threadIdx.x;                                             // RECOMPUTE
  double* const sGq = reinterpret_cast<double*>(smraw + C::off_gq) + threadIdx.x; // RECOMPUTE
  const int32_t* sE = reinterpret_cast<const int32_t*>(smraw + C::off_enc);
  double* su = reinterpret_cast<double*>(smraw + C::off_su);
  double* sf = reinterpret_cast<double*>(smraw + C::off_sf);
  uint64_t* fullG = reinterpret_cast<uint64_t*>(smraw + C::off_bar);
  uint64_t* fullE = fullG + R;

  const int tid = threadIdx.x;
  const int cl = tid / n;
  const int k = tid - cl * n;
  const bool in_block = cl < CPB;
  const int cls = in_block ? cl : 0;
  const int my_nb = ((int)blockIdx.x < nbatch) ? (nbatch - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int total_planes = my_nb * n;

  uint64_t pol = 0;
  if (tid == 0)
  {
    for (int s = 0; s < R + 2; ++s)
      mbar_init(&fullG[s], 1);
    mbar_fence_init();
    pol = policy_evict_first();
  }
  __syncthreads();

  // producer state (thread 0 only): next plane to issue
  int issue_t = 0;
  auto issue_plane = [&](int t)
  {
    const int it = t / n, i = t - it * n;
    const long long gb = batch0 + blockIdx.x + (long long)it * gridDim.x;
    const int s = t % R;
    mbar_expect_tx(&fullG[s], C::plane_bytes);
    bulk_g2s(sG + (size_t)s * C::plane_doubles, G + (gb * n2 + (long long)i * n) * 6 * S, C::plane_bytes,
             &fullG[s], pol);
  };
  auto issue_enc = [&](int it)
  {
    const long long gb = batch0 + blockIdx.x + (long long)it * gridDim.x;
    const int eb = it & 1;
    mbar_expect_tx(&fullE[eb], C::enc_bytes);
    bulk_g2s(const_cast<int32_t*>(sE) + eb * (n2 * SE), enc + gb * (long long)(n2 * SE), C::enc_bytes, &fullE[eb], pol);
  };
  if (tid == 0 && my_nb > 0)
  {
    issue_enc(0);
    if constexpr (!RECOMPUTE)
      for (; issue_t < R && issue_t < total_planes; ++issue_t)
        issue_plane(issue_t);
  }

  double Dk[n], DTk[n];
#pragma unroll
  for (int l = 0; l < n; ++l)
  {
    Dk[l] = c_D[P][k * n + l];
    DTk[l] = c_D[P][l * n + k];
  }
  const double zeta = c_pts[P][k], wk = c_wts[P][k]; // RECOMPUTE

  int stage = 0;
  uint32_t stage_parity = 0;
  for (int it = 0; it < my_nb; ++it)
  {
    const int b = blockIdx.x + it * gridDim.x;
    const int pl = b * CPB + cl;
    const bool active = in_block && pl < count;

    const int eb = it & 1;
    mbar_wait(&fullE[eb], (it >> 1) & 1);
    const int32_t* dE = sE + eb * (n2 * SE) + tid; // this thread's n2 encoded dofs
    double u[n2];
    double kap = 0.0;
    if constexpr (RECOMPUTE)
    { // this thread's plane zeta of the cell; the previous batch's reads of sJ / sGq were its own, earlier
      TrilinearMonomials M;
      M.load(xgeom, active ? geom_dofmap + (long long)perm[cell0 + pl] * 8 : nullptr);
      JacobianAtZeta jac;
      jac.init(M, zeta);
      jac.store(sJ, TPB);
    }
    if (active)
    {
      kap = kappa[perm[cell0 + pl]];
#pragma unroll
      for (int a = 0; a < n2; ++a)
      {
        const int da = dE[a * SE];
        const int idx = da < 0 ? ~da : da;
        const double xv = x[idx];
        if (da < 0)
          y[idx] = xv; // Dirichlet row: y = x (src/laplacian.hpp:273-274)
        u[a] = da < 0 ? 0.0 : xv;
      }
    }
    else
    {
#pragma unroll
      for (int a = 0; a < n2; ++a)
        u[a] = 0.0;
    }
    if (in_block)
    {
#pragma unroll
      for (int j = 0; j < n; ++j)
        su[cl * CS + j * KP + k] = u[j];
    }
    __syncthreads(); // z-rows of plane 0 are visible; the other dofmap buffer (batch it-1) is free
    if (tid == 0 && it + 1 < my_nb)
      issue_enc(it + 1);

    double acc[n2];
#pragma unroll
    for (int a = 0; a < n2; ++a)
      acc[a] = 0.0;

#pragma unroll
    for (int i = 0; i < n; ++i)
    {
      if constexpr (!RECOMPUTE)
        mbar_wait(&fullG[stage], stage_parity);
      const double* gs = RECOMPUTE ? sGq : sG + (size_t)stage * C::plane_doubles + tid;
      const double* sup = su + ((i & 1) * CPB + cls) * CS;
      double* sfz = sf + ((i & 1) * CPB + cls) * CS;
      if constexpr (RECOMPUTE)
      { // G at the points (i, j, k), j = 0..n-1, one point at a time: the slab (u, acc) keeps the registers
        const JacobianAtZeta::Plane jp = JacobianAtZeta::plane(sJ, TPB, c_pts[P][i]);
        const double wik = c_wts[P][i] * wk;
#pragma unroll 1
        for (int j = 0; j < n; ++j)
        {
          double J[3][3], g[6];
          JacobianAtZeta::at(sJ, TPB, jp, c_pts[P][j], J);
          g_from_jacobian(J, literal_detj, wik * c_wts[P][j], g);
#pragma unroll
          for (int c = 0; c < 6; ++c)
            sGq[(j * 6 + c) * TPB] = g[c];
        }
      }
      double fz[n];
#pragma unroll
      for (int j = 0; j < n; ++j)
      {
        double gx = 0.0, gy = 0.0, gz = 0.0;
        const double2* row = reinterpret_cast<const double2*>(sup + j * KP);
#pragma unroll
        for (int l2 = 0; l2 < KP / 2; ++l2)
        {
          const double2 r = row[l2];
          gz = fma(Dk[2 * l2], r.x, gz);
          if (2 * l2 + 1 < n)
            gz = fma(Dk[2 * l2 + 1], r.y, gz);
        }
#pragma unroll
        for (int l = 0; l < n; ++l)
        {
          gx = fma(c_D[P][i * n + l], u[l * n + j], gx);
          gy = fma(c_D[P][j * n + l], u[i * n + l], gy);
        }
        const double g0 = gs[(j * 6 + 0) * GS], g1 = gs[(j * 6 + 1) * GS], g2 = gs[(j * 6 + 2) * GS];
        const double g3 = gs[(j * 6 + 3) * GS], g4 = gs[(j * 6 + 4) * GS], g5 = gs[(j * 6 + 5) * GS];
        const double fx = kap * (g0 * gx + g1 * gy + g2 * gz);
        const double fy = kap * (g1 * gx + g3 * gy + g4 * gz);
        fz[j] = kap * (g2 * gx + g4 * gy + g5 * gz);
#pragma unroll
        for (int l = 0; l < n; ++l)
        {
          acc[l * n + j] = fma(c_D[P][i * n + l], fx, acc[l * n + j]);
          acc[i * n + l] = fma(c_D[P][j * n + l], fy, acc[i * n + l]);
        }
      }
      if (in_block)
      {
#pragma unroll
        for (int j = 0; j < n; ++j)
          sfz[j * KP + k] = fz[j];
        if (i + 1 < n)
        {
          double* sun = su + (((i + 1) & 1) * CPB + cl) * CS;
#pragma unroll
          for (int j = 0; j < n; ++j)
            sun[j * KP + k] = u[(i + 1) * n + j];
        }
      }
      __syncthreads(); // geometry stage is consumed; fz rows and next z-rows are visible
      if constexpr (!RECOMPUTE)
      {
        if (tid == 0)
        {
          if (issue_t < total_planes)
            issue_plane(issue_t++);
        }
        if (++stage == R)
        {
          stage = 0;
          stage_parity ^= 1u;
        }
      }
#pragma unroll
      for (int j = 0; j < n; ++j)
      {
        const double2* row = reinterpret_cast<const double2*>(sfz + j * KP);
        double t = 0.0;
#pragma unroll
        for (int q2 = 0; q2 < KP / 2; ++q2)
        {
          const double2 r = row[q2];
          t = fma(DTk[2 * q2], r.x, t);
          if (2 * q2 + 1 < n)
            t = fma(DTk[2 * q2 + 1], r.y, t);
        }
        acc[i * n + j] += t;
      }
    }
    if (active)
    {
#pragma unroll
      for (int a = 0; a < n2; ++a)
      {
        const int da = dE[a * SE];
        if (da >= 0)
          atomicAdd(&y[da], acc[a]);
      }
    }
  }
}

template <int P, int TPB, bool RECOMPUTE = false>
struct TmaApply
{
  using C = TmaCfg<P, TPB, RECOMPUTE>;
  static constexpr bool cell_geometry = false;
  static constexpr int cpb = C::cpb;
  static void name(char* s, int cap)
  {
    if (RECOMPUTE)
      snprintf(s, cap, "k_apply_tma<%d,%d,recomputed>", P, TPB);
    else
      snprintf(s, cap, "k_apply_tma<%d,%d,%d>", P, TPB, C::R);
  }
  static void launch(pmgx_ctx* c, cudaStream_t st, const ApplyArgs& a)
  {
    launch_batched<k_apply_tma<P, TPB, RECOMPUTE>, C>(c, st, a, "k_apply_tma", a.xgeom, a.geom_dofmap, a.literal_detj);
  }
};

// ------------------------------------------------ the affine-geometry apply kernel --
// On a cell whose trilinear map is affine (every cell of a box / parallelepiped mesh, i.e. all
// the benchmark meshes) J is constant, so G(q) = w_q * Gc with ONE 6-vector Gc = K K^T / det J per
// cell: the 48 B per quadrature point that make up 79 % of the streamed bytes of the apply collapse
// to 48 B per cell.  When ALL cells of an operator pass the affinity test at create
// (k_cell_geometry, tolerance 1e-13 h) this kernel replaces k_apply_tma: same thread mapping and
// arithmetic (thread = z-index of a cell, (ix,iy) slab in registers, z contraction through
// shared memory), but nothing is streamed except the encoded dofmap (cp.async.bulk double
// buffer); the kernel is then bound by the gather / atomic traffic of x and y in L2, not by HBM.
// Meshes with any non-affine cell keep the streamed-G kernels; PMGX_LAP_STREAM_G forces them.
template <int P, int TPB>
struct AffCfg
{
  static constexpr int n = P + 1;
  static constexpr int n2 = n * n;
  static constexpr int tpb = TPB;
  static constexpr int cpb = tpb / n;
  static constexpr int SE = (cpb * n + 3) & ~3;
  static constexpr int kp = n + (n & 1);
  static constexpr int cs = ((n * kp / 2) & 1) ? n * kp : n * kp + 2;
  static constexpr uint32_t enc_bytes = n2 * SE * sizeof(int32_t);
  static constexpr int buf_doubles = 2 * cpb * cs;
  static constexpr size_t off_su = 2 * (size_t)enc_bytes;
  static constexpr size_t off_sf = off_su + (size_t)buf_doubles * sizeof(double);
  static constexpr size_t off_bar = off_sf + (size_t)buf_doubles * sizeof(double);
  static constexpr size_t smem = off_bar + 2 * sizeof(uint64_t);
  static constexpr int minb = P <= 2 ? 6 : (TPB <= 64 ? 4 : 2);
};

template <int P, int TPB>
__global__ void __launch_bounds__(TPB, AffCfg<P, TPB>::minb)
k_apply_affine(const double* __restrict__ x, double* __restrict__ y, const double* __restrict__ Gc,
               const int32_t* __restrict__ enc, const int32_t* __restrict__ perm,
               const double* __restrict__ kappa, long long batch0, int cell0, int count, int nbatch)
{
  using C = AffCfg<P, TPB>;
  constexpr int n = C::n, n2 = C::n2, CPB = C::cpb, SE = C::SE, KP = C::kp, CS = C::cs;
  extern __shared__ __align__(128) unsigned char smraw[];
  const int32_t* sE = reinterpret_cast<const int32_t*>(smraw);
  double* su = reinterpret_cast<double*>(smraw + C::off_su);
  double* sf = reinterpret_cast<double*>(smraw + C::off_sf);
  uint64_t* fullE = reinterpret_cast<uint64_t*>(smraw + C::off_bar);

  const int tid = threadIdx.x;
  const int cl = tid / n;
  const int k = tid - cl * n;
  const bool in_block = cl < CPB;
  const int cls = in_block ? cl : 0;
  const int my_nb = ((int)blockIdx.x < nbatch) ? (nbatch - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

  uint64_t pol = 0;
  if (tid == 0)
  {
    mbar_init(&fullE[0], 1);
    mbar_init(&fullE[1], 1);
    mbar_fence_init();
    pol = policy_evict_first();
  }
  __syncthreads();
  auto issue_enc = [&](int it)
  {
    const long long gb = batch0 + blockIdx.x + (long long)it * gridDim.x;
    mbar_expect_tx(&fullE[it & 1], C::enc_bytes);
    bulk_g2s(const_cast<int32_t*>(sE) + (it & 1) * (n2 * SE), enc + gb * (long long)(n2 * SE), C::enc_bytes,
             &fullE[it & 1], pol);
  };
  if (tid == 0 && my_nb > 0)
    issue_enc(0);

  double Dk[n], DTk[n];
#pragma unroll
  for (int l = 0; l < n; ++l)
  {
    Dk[l] = c_D[P][k * n + l];
    DTk[l] = c_D[P][l * n + k];
  }
  const double wk = c_wts[P][k];

  for (int it = 0; it < my_nb; ++it)
  {
    const int b = blockIdx.x + it * gridDim.x;
    const int pl = b * CPB + cl;
    const bool active = in_block && pl < count;

    mbar_wait(&fullE[it & 1], (it >> 1) & 1);
    const int32_t* dE = sE + (it & 1) * (n2 * SE) + tid;
    double u[n2];
    double g[6];
    if (active)
    {
      const double kw = kappa[perm[cell0 + pl]] * wk; // kappa re-read on every apply (src/laplacian.hpp:230)
      const double* gp = Gc + (size_t)(cell0 + pl) * 6;
#pragma unroll
      for (int c = 0; c < 6; ++c)
        g[c] = gp[c] * kw;
#pragma unroll
      for (int a = 0; a < n2; ++a)
      {
        const int da = dE[a * SE];
        const int idx = da < 0 ? ~da : da;
        const double xv = x[idx];
        if (da < 0)
          y[idx] = xv; // Dirichlet row: y = x (src/laplacian.hpp:273-274)
        u[a] = da < 0 ? 0.0 : xv;
      }
    }
    else
    {
#pragma unroll
      for (int c = 0; c < 6; ++c)
        g[c] = 0.0;
#pragma unroll
      for (int a = 0; a < n2; ++a)
        u[a] = 0.0;
    }
    if (in_block)
    {
#pragma unroll
      for (int j = 0; j < n; ++j)
        su[cl * CS + j * KP + k] = u[j];
    }
    __syncthreads(); // z-rows of plane 0 are visible; the other dofmap buffer (batch it-1) is free
    if (tid == 0 && it + 1 < my_nb)
      issue_enc(it + 1);

    double acc[n2];
#pragma unroll
    for (int a = 0; a < n2; ++a)
      acc[a] = 0.0;

#pragma unroll
    for (int i = 0; i < n; ++i)
    {
      const double* sup = su + ((i & 1) * CPB + cls) * CS;
      double* sfz = sf + ((i & 1) * CPB + cls) * CS;
      double fz[n];
#pragma unroll
      for (int j = 0; j < n; ++j)
      {
        double gx = 0.0, gy = 0.0, gz = 0.0;
        const double2* row = reinterpret_cast<const double2*>(sup + j * KP);
#pragma unroll
        for (int l2 = 0; l2 < n / 2; ++l2)
        {
          const double2 r = row[l2];
          gz = fma(Dk[2 * l2], r.x, gz);
          gz = fma(Dk[2 * l2 + 1], r.y, gz);
        }
        if (n & 1) // odd n: the last entry alone (a 64-bit load: half the wavefronts of a padded 128-bit one)
          gz = fma(Dk[n - 1], sup[j * KP + n - 1], gz);
#pragma unroll
        for (int l = 0; l < n; ++l)
        {
          gx = fma(c_D[P][i * n + l], u[l * n + j], gx);
          gy = fma(c_D[P][j * n + l], u[i * n + l], gy);
        }
        const double wij = c_wts[P][i] * c_wts[P][j]; // G(q) = w_i w_j w_k Gc
        const double fx = wij * (g[0] * gx + g[1] * gy + g[2] * gz);
        const double fy = wij * (g[1] * gx + g[3] * gy + g[4] * gz);
        fz[j] = wij * (g[2] * gx + g[4] * gy + g[5] * gz);
#pragma unroll
        for (int l = 0; l < n; ++l)
        {
          acc[l * n + j] = fma(c_D[P][i * n + l], fx, acc[l * n + j]);
          acc[i * n + l] = fma(c_D[P][j * n + l], fy, acc[i * n + l]);
        }
      }
      if (in_block)
      {
#pragma unroll
        for (int j = 0; j < n; ++j)
          sfz[j * KP + k] = fz[j];
        if (i + 1 < n)
        {
          double* sun = su + (((i + 1) & 1) * CPB + cl) * CS;
#pragma unroll
          for (int j = 0; j < n; ++j)
            sun[j * KP + k] = u[(i + 1) * n + j];
        }
      }
      __syncthreads(); // fz rows and the next z-rows are visible
#pragma unroll
      for (int j = 0; j < n; ++j)
      {
        const double2* row = reinterpret_cast<const double2*>(sfz + j * KP);
        double t = 0.0;
#pragma unroll
        for (int q2 = 0; q2 < n / 2; ++q2)
        {
          const double2 r = row[q2];
          t = fma(DTk[2 * q2], r.x, t);
          t = fma(DTk[2 * q2 + 1], r.y, t);
        }
        if (n & 1)
          t = fma(DTk[n - 1], sfz[j * KP + n - 1], t);
        acc[i * n + j] += t;
      }
    }
    if (active)
    {
#pragma unroll
      for (int a = 0; a < n2; ++a)
      {
        const int da = dE[a * SE];
        if (da >= 0)
          atomicAdd(&y[da], acc[a]);
      }
    }
  }
}

template <int P, int TPB>
struct AffineApply
{
  using C = AffCfg<P, TPB>;
  static constexpr bool cell_geometry = true;
  static constexpr int cpb = C::cpb;
  static void name(char* s, int cap) { snprintf(s, cap, "k_apply_affine<%d,%d>", P, TPB); }
  static void launch(pmgx_ctx* c, cudaStream_t st, const ApplyArgs& a)
  {
    launch_batched<k_apply_affine<P, TPB>, C>(c, st, a, "k_apply_affine");
  }
};

// Shuffle variant of the affine kernel: a warp holds 32/n whole cells (lanes beyond that idle), so
// the z contractions are warp shuffles from the n lanes of the thread's own cell -- no shared-memory
// rows, no block barrier per plane.  ncu on the shared-memory variant at P4: L1/shared data pipe 78 %
// busy with 20 %-efficient broadcast reads; n double shuffles move the same data in ~40 % fewer
// pipe cycles and the warps of a CTA no longer wait for each other.
template <int P, int TPB>
struct AffShCfg
{
  static constexpr int n = P + 1;
  static constexpr int n2 = n * n;
  static constexpr int tpb = TPB;
  static constexpr int cpw = 32 / n;               // cells per warp
  static constexpr int cpb = (TPB / 32) * cpw;     // cells per batch
  static constexpr int SE = (cpb * n + 3) & ~3;
  static constexpr uint32_t enc_bytes = n2 * SE * sizeof(int32_t);
  static constexpr size_t off_bar = 2 * (size_t)enc_bytes;
  static constexpr size_t smem = off_bar + 2 * sizeof(uint64_t);
  static constexpr int minb = P <= 2 ? 6 : (TPB <= 64 ? 4 : 2);
};

template <int P, int TPB>
__global__ void __launch_bounds__(TPB, AffShCfg<P, TPB>::minb)
k_apply_affine_shfl(const double* __restrict__ x, double* __restrict__ y, const double* __restrict__ Gc,
                    const int32_t* __restrict__ enc, const int32_t* __restrict__ perm,
                    const double* __restrict__ kappa, long long batch0, int cell0, int count, int nbatch)
{
  using C = AffShCfg<P, TPB>;
  constexpr int n = C::n, n2 = C::n2, CPB = C::cpb, CPW = C::cpw, SE = C::SE;
  extern __shared__ __align__(128) unsigned char smraw[];
  const int32_t* sE = reinterpret_cast<const int32_t*>(smraw);
  uint64_t* fullE = reinterpret_cast<uint64_t*>(smraw + C::off_bar);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int cw = lane / n;                 // cell within the warp
  const int k = lane - cw * n;             // iz
  const bool lane_ok = cw < CPW;
  const int cl = warp * CPW + (lane_ok ? cw : 0);
  const int base = (lane_ok ? cw : 0) * n; // first lane of this thread's cell
  const int slot = cl * n + (lane_ok ? k : 0);
  const int my_nb = ((int)blockIdx.x < nbatch) ? (nbatch - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

  uint64_t pol = 0;
  if (tid == 0)
  {
    mbar_init(&fullE[0], 1);
    mbar_init(&fullE[1], 1);
    mbar_fence_init();
    pol = policy_evict_first();
  }
  __syncthreads();
  auto issue_enc = [&](int it)
  {
    const long long gb = batch0 + blockIdx.x + (long long)it * gridDim.x;
    mbar_expect_tx(&fullE[it & 1], C::enc_bytes);
    bulk_g2s(const_cast<int32_t*>(sE) + (it & 1) * (n2 * SE), enc + gb * (long long)(n2 * SE), C::enc_bytes,
             &fullE[it & 1], pol);
  };
  if (tid == 0 && my_nb > 0)
  {
    issue_enc(0);
    if (my_nb > 1)
      issue_enc(1);
  }

  const int kk = lane_ok ? k : 0;
  double Dk[n], DTk[n];
#pragma unroll
  for (int l = 0; l < n; ++l)
  {
    Dk[l] = c_D[P][kk * n + l];
    DTk[l] = c_D[P][l * n + kk];
  }
  const double wk = c_wts[P][kk];

  for (int it = 0; it < my_nb; ++it)
  {
    const int b = blockIdx.x + it * gridDim.x;
    const int pl = b * CPB + cl;
    const bool active = lane_ok && pl < count;

    mbar_wait(&fullE[it & 1], (it >> 1) & 1);
    const int32_t* dE = sE + (it & 1) * (n2 * SE) + slot;
    double u[n2];
    double g[6];
    if (active)
    {
      const double kw = kappa[perm[cell0 + pl]] * wk; // kappa re-read on every apply (src/laplacian.hpp:230)
      const double* gp = Gc + (size_t)(cell0 + pl) * 6;
#pragma unroll
      for (int c = 0; c < 6; ++c)
        g[c] = gp[c] * kw;
#pragma unroll
      for (int a = 0; a < n2; ++a)
      {
        const int da = dE[a * SE];
        const int idx = da < 0 ? ~da : da;
        const double xv = x[idx];
        if (da < 0)
          y[idx] = xv; // Dirichlet row: y = x (src/laplacian.hpp:273-274)
        u[a] = da < 0 ? 0.0 : xv;
      }
    }
    else
    {
#pragma unroll
      for (int c = 0; c < 6; ++c)
        g[c] = 0.0;
#pragma unroll
      for (int a = 0; a < n2; ++a)
        u[a] = 0.0;
    }
    double acc[n2];
#pragma unroll
    for (int a = 0; a < n2; ++a)
      acc[a] = 0.0;

#pragma unroll
    for (int i = 0; i < n; ++i)
    {
#pragma unroll
      for (int j = 0; j < n; ++j)
      {
        double gx = 0.0, gy = 0.0, gz = 0.0;
        const double uij = u[i * n + j];
#pragma unroll
        for (int l = 0; l < n; ++l)
        {
          gz = fma(Dk[l], __shfl_sync(0xffffffffu, uij, base + l), gz);
          gx = fma(c_D[P][i * n + l], u[l * n + j], gx);
          gy = fma(c_D[P][j * n + l], u[i * n + l], gy);
        }
        const double wij = c_wts[P][i] * c_wts[P][j]; // G(q) = w_i w_j w_k Gc
        const double fx = wij * (g[0] * gx + g[1] * gy + g[2] * gz);
        const double fy = wij * (g[1] * gx + g[3] * gy + g[4] * gz);
        const double fz = wij * (g[2] * gx + g[4] * gy + g[5] * gz);
        double t = 0.0;
#pragma unroll
        for (int q = 0; q < n; ++q)
          t = fma(DTk[q], __shfl_sync(0xffffffffu, fz, base + q), t);
#pragma unroll
        for (int l = 0; l < n; ++l)
        {
          acc[l * n + j] = fma(c_D[P][i * n + l], fx, acc[l * n + j]);
          acc[i * n + l] = fma(c_D[P][j * n + l], fy, acc[i * n + l]);
        }
        acc[i * n + j] += t;
      }
    }
    if (active)
    {
#pragma unroll
      for (int a = 0; a < n2; ++a)
      {
        const int da = dE[a * SE];
        if (da >= 0)
          atomicAdd(&y[da], acc[a]);
      }
    }
    // every thread is done with this batch's dofmap buffer before the one after next may land in it
    __syncthreads();
    if (tid == 0 && it + 2 < my_nb)
      issue_enc(it + 2);
  }
}

template <int P, int TPB>
struct AffineShflApply
{
  using C = AffShCfg<P, TPB>;
  static constexpr bool cell_geometry = true;
  static constexpr int cpb = C::cpb;
  static void name(char* s, int cap) { snprintf(s, cap, "k_apply_affine_shfl<%d,%d>", P, TPB); }
  static void launch(pmgx_ctx* c, cudaStream_t st, const ApplyArgs& a)
  {
    launch_batched<k_apply_affine_shfl<P, TPB>, C>(c, st, a, "k_apply_affine_shfl");
  }
};


// ---------------------------------------- the re-slabbed affine-geometry apply kernel --
// Same thread mapping as k_apply_affine (thread t of a cell holds the (ix,iy) slab at iz = t in
// registers, x and y contractions are register FMAs), but the z direction no longer re-reads every
// z-row of the element n times as a broadcast (2 n^3 + 2 n^2 shared-memory doubles per thread; ncu:
// L1/shared data pipe 78 % busy at 42 % FP64, profiles/r1_apply_p4_affine.txt).  Instead the data is
// RE-SLABBED: every value crosses shared memory once per phase, written by the thread that owns it
// and read by the thread that needs it --
//   1. u(i,j,t)        -> thread j reads the slab u(i,j,.) and forms gz(i,j,l) = sum_m D[l][m] u(i,j,m)
//   2. gz(i,j,l)       -> thread l reads gz(.,.,l): all three gradients at its points; G-transform;
//                         x and y transposed contractions into the register accumulator
//   3. fz(i,j,t)       -> thread j reads fz(i,j,.) and forms az(i,j,l) = sum_q D[q][l] fz(i,j,q)
//   4. az(i,j,l)       -> thread l adds az(.,.,l) to its accumulator
// 8 n^2 doubles per thread instead of 2 n^3 + 2 n^2 (P4: 200 vs 300; P6: 392 vs 784), no broadcast
// reads, and one CTA barrier per batch instead of n + 1: a warp holds 32 / n WHOLE cells (the lanes
// beyond that idle), so every exchange stays inside a warp and the phases are separated by
// __syncwarp(): the warps of a CTA run free of each other (with 8-10 warps per SM a CTA barrier per
// phase leaves the schedulers empty).  Strides: slab stride SS = 1 (mod 16) and cell
// stride CS = n (mod 16) doubles make the 8-byte bank of BOTH access patterns (unit stride in t when
// writing, stride SS in t when reading) equal to lane + const: every 64-bit access is conflict-free.
template <int P, int TPB>
struct Aff2Cfg
{
  static constexpr int n = P + 1;
  static constexpr int n2 = n * n;
  static constexpr int tpb = TPB;
  static constexpr int cpw = 32 / n;               // cells per warp
  static constexpr int cpb = (TPB / 32) * cpw;     // cells per batch
  static constexpr int SE = (cpb * n + 3) & ~3;
  static constexpr int ss = ((n2 - 1 + 15) / 16) * 16 + 1;                 // >= n2, = 1 mod 16
  static constexpr int cs = ((n * ss - n + 15) / 16) * 16 + n;             // >= n * ss, = n mod 16
  static constexpr uint32_t enc_bytes = n2 * SE * sizeof(int32_t);
  static constexpr int buf_doubles = cpb * cs;
  static constexpr size_t off_a = 2 * (size_t)enc_bytes;
  static constexpr size_t off_b = off_a + (size_t)buf_doubles * sizeof(double);
  static constexpr size_t off_bar = off_b + (size_t)buf_doubles * sizeof(double);
  static constexpr size_t smem = off_bar + 2 * sizeof(uint64_t);
  static constexpr int minb = P <= 2 ? 6 : (P <= 4 ? 4 : 2);
};

template <int P, int TPB>
__global__ void __launch_bounds__(TPB, Aff2Cfg<P, TPB>::minb)
k_apply_affine2(const double* __restrict__ x, double* __restrict__ y, const double* __restrict__ Gc,
                const int32_t* __restrict__ enc, const int32_t* __restrict__ perm,
                const double* __restrict__ kappa, long long batch0, int cell0, int count, int nbatch)
{
  using C = Aff2Cfg<P, TPB>;
  constexpr int n = C::n, n2 = C::n2, CPB = C::cpb, SE = C::SE, SS = C::ss, CS = C::cs;
  extern __shared__ __align__(128) unsigned char smraw[];
  const int32_t* sE = reinterpret_cast<const int32_t*>(smraw);
  double* sA = reinterpret_cast<double*>(smraw + C::off_a);
  double* sB = reinterpret_cast<double*>(smraw + C::off_b);
  uint64_t* fullE = reinterpret_cast<uint64_t*>(smraw + C::off_bar);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int cw = lane / n;
  const bool in_block = cw < C::cpw;
  const int cl = warp * C::cpw + (in_block ? cw : 0);
  const int t = in_block ? lane - cw * n : 0;
  const int cls = in_block ? cl : 0;
  const int slot = cls * n + t;
  const int my_nb = ((int)blockIdx.x < nbatch) ? (nbatch - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

  uint64_t pol = 0;
  if (tid == 0)
  {
    mbar_init(&fullE[0], 1);
    mbar_init(&fullE[1], 1);
    mbar_fence_init();
    pol = policy_evict_first();
  }
  __syncthreads();
  auto issue_enc = [&](int it)
  {
    const long long gb = batch0 + blockIdx.x + (long long)it * gridDim.x;
    mbar_expect_tx(&fullE[it & 1], C::enc_bytes);
    bulk_g2s(const_cast<int32_t*>(sE) + (it & 1) * (n2 * SE), enc + gb * (long long)(n2 * SE), C::enc_bytes,
             &fullE[it & 1], pol);
  };
  if (tid == 0 && my_nb > 0)
    issue_enc(0);

  const double wt = c_wts[P][t];
  // writer view: element (slab s, row r) of this thread's z-index; reader view: this thread's slab
  double* const wA = sA + cls * CS + t;
  double* const wB = sB + cls * CS + t;
  const double* const rA = sA + cls * CS + t * SS;
  const double* const rB = sB + cls * CS + t * SS;

  for (int it = 0; it < my_nb; ++it)
  {
    const int b = blockIdx.x + it * gridDim.x;
    const int pl = b * CPB + cl;
    const bool active = in_block && pl < count;

    // the only CTA barrier of a batch: every warp is done with the dofmap buffer the next load will overwrite
    __syncthreads();
    if (tid == 0 && it + 1 < my_nb)
      issue_enc(it + 1);
    mbar_wait(&fullE[it & 1], (it >> 1) & 1);
    const int32_t* dE = sE + (it & 1) * (n2 * SE) + slot;
    double u[n2];
    double g[6];
    if (active)
    {
      const double kw = kappa[perm[cell0 + pl]] * wt; // kappa re-read on every apply (src/laplacian.hpp:230)
      const double* gp = Gc + (size_t)(cell0 + pl) * 6;
#pragma unroll
      for (int c = 0; c < 6; ++c)
        g[c] = gp[c] * kw;
#pragma unroll
      for (int a = 0; a < n2; ++a)
      {
        const int da = dE[a * SE];
        const int idx = da < 0 ? ~da : da;
        const double xv = x[idx];
        if (da < 0)
          y[idx] = xv; // Dirichlet row: y = x (src/laplacian.hpp:273-274)
        u[a] = da < 0 ? 0.0 : xv;
      }
    }
    else
    {
#pragma unroll
      for (int c = 0; c < 6; ++c)
        g[c] = 0.0;
#pragma unroll
      for (int a = 0; a < n2; ++a)
        u[a] = 0.0;
    }
    // phase 1: u(i,j,t) -> A[slab j][i][t]
    if (in_block)
    {
#pragma unroll
      for (int i = 0; i < n; ++i)
#pragma unroll
        for (int j = 0; j < n; ++j)
          wA[j * SS + i * n] = u[i * n + j];
    }
    __syncwarp();
    // phase 2: slab j = t: gz(i,t,l) = sum_m D[l][m] u(i,t,m) -> B[slab l][i][t]
#pragma unroll
    for (int i = 0; i < n; ++i)
    {
      double v[n];
#pragma unroll
      for (int m = 0; m < n; ++m)
        v[m] = rA[i * n + m];
#pragma unroll
      for (int l = 0; l < n; ++l)
      {
        double s = 0.0;
#pragma unroll
        for (int m = 0; m < n; ++m)
          s = fma(c_D[P][l * n + m], v[m], s);
        if (in_block)
          wB[l * SS + i * n] = s;
      }
    }
    __syncwarp();
    // phase 3: all three gradients at the points (i,j,t); transform; x / y transposed contractions;
    // fz(i,j,t) -> A[slab j][i][t]
    double acc[n2];
#pragma unroll
    for (int a = 0; a < n2; ++a)
      acc[a] = 0.0;
#pragma unroll
    for (int i = 0; i < n; ++i)
#pragma unroll
      for (int j = 0; j < n; ++j)
      {
        double gx = 0.0, gy = 0.0;
        const double gz = rB[i * n + j];
#pragma unroll
        for (int l = 0; l < n; ++l)
        {
          gx = fma(c_D[P][i * n + l], u[l * n + j], gx);
          gy = fma(c_D[P][j * n + l], u[i * n + l], gy);
        }
        const double wij = c_wts[P][i] * c_wts[P][j]; // G(q) = w_i w_j w_k Gc
        const double fx = wij * (g[0] * gx + g[1] * gy + g[2] * gz);
        const double fy = wij * (g[1] * gx + g[3] * gy + g[4] * gz);
        const double fz = wij * (g[2] * gx + g[4] * gy + g[5] * gz);
#pragma unroll
        for (int l = 0; l < n; ++l)
        {
          acc[l * n + j] = fma(c_D[P][i * n + l], fx, acc[l * n + j]);
          acc[i * n + l] = fma(c_D[P][j * n + l], fy, acc[i * n + l]);
        }
        if (in_block)
          wA[j * SS + i * n] = fz;
      }
    __syncwarp();
    // phase 4: slab j = t: az(i,t,l) = sum_q D[q][l] fz(i,t,q) -> B[slab l][i][t]
#pragma unroll
    for (int i = 0; i < n; ++i)
    {
      double v[n];
#pragma unroll
      for (int q = 0; q < n; ++q)
        v[q] = rA[i * n + q];
#pragma unroll
      for (int l = 0; l < n; ++l)
      {
        double s = 0.0;
#pragma unroll
        for (int q = 0; q < n; ++q)
          s = fma(c_D[P][q * n + l], v[q], s);
        if (in_block)
          wB[l * SS + i * n] = s;
      }
    }
    __syncwarp();
    // phase 5: acc(i,j,t) += az(i,j,t); scatter
    if (active)
    {
#pragma unroll
      for (int a = 0; a < n2; ++a)
      {
        const int da = dE[a * SE];
        if (da >= 0)
          atomicAdd(&y[da], acc[a] + rB[a]);
      }
    }
    __syncwarp(); // B is rewritten in the next batch's phase 2 only after this warp's reads above
  }
}

template <int P, int TPB>
struct Affine2Apply
{
  using C = Aff2Cfg<P, TPB>;
  static constexpr bool cell_geometry = true;
  static constexpr int cpb = C::cpb;
  static void name(char* s, int cap) { snprintf(s, cap, "k_apply_affine2<%d,%d,warp-local>", P, TPB); }
  static void launch(pmgx_ctx* c, cudaStream_t st, const ApplyArgs& a)
  {
    launch_batched<k_apply_affine2<P, TPB>, C>(c, st, a, "k_apply_affine2");
  }
};

#include "laplacian_mma.cuh"

// ------------------------------------------------------------- the kernel per degree --
// Affine: every cell of the operator passed the affinity test at create (k_cell_geometry); Streamed: G per
// quadrature point (any non-affine cell, or PMGX_LAP_STREAM_G).  The choices were measured at 100 M dofs:
// * threads per CTA of the affine slab kernels, 128 vs 64: P1 3.45 vs 4.07 ms, P2 1.67 vs 1.79, P3 1.61 vs 1.54,
//   P4 1.34 vs 1.28, P5 1.20 vs 1.19, P6 2.06 vs 2.03 (P3 re-slab kernel: 1.201 / 1.202 ms at 64 / 128);
// * z contraction by warp shuffles (k_apply_affine_shfl) vs shared-memory rows: P1 3.52 vs 3.45 ms, P2 1.58 vs
//   1.67, P3 1.63 vs 1.54, P4 1.36 vs 1.28, P5 1.57 vs 1.19, P6 2.27 vs 2.03 -- double shuffles cost two issue
//   slots each and only pay where the element is small;
// * re-slabbed z direction (k_apply_affine2) vs broadcast rows: P1 4.16 vs 3.44 ms, P2 1.76 vs 1.58, P3 1.20 vs
//   1.54, P4 1.41 vs 1.28, P5 2.40 vs 1.19, P6 3.09 vs 2.03: it halves the shared-memory wavefronts (ncu: L1/shared
//   pipe 78 -> 53 %) but both kernels sit at 2 warps per scheduler with fixed-latency (DFMA dependency) stalls on
//   top, so it only wins where its register count drops far enough to matter (P3);
// * streamed G: threads per CTA of k_apply_tma, the winners of a sweep over {64, 128} threads x {2, 3, 4}
//   geometry planes in flight on a B200;
// * P6 / P7: the FP64 tensor-core kernel against the slab kernels, see laplacian_mma.cuh;
// * P8: the column kernel; the slab kernels keep 2 (P+1)^2 doubles in registers per thread (measured: P7 53 % vs
//   47 %, P8 24 % vs 27 %) and n = 9 fits no 8-wide tensor-core tile.  It has no affine variant, so the affinity
//   test is skipped and is_affine() stays 0.
// * Recompute (PMGX_LAP_RECOMPUTE_G): each family's geometry-from-vertices variant, with the thread mapping and the
//   launch configuration of its streamed-G kernel.
template <int P>
struct ApplyKernels;
// clang-format off
template <> struct ApplyKernels<1> { using Affine = AffineApply<1, 128>;     using Streamed = TmaApply<1, 64>;  using Recompute = TmaApply<1, 64, true>; };
template <> struct ApplyKernels<2> { using Affine = AffineShflApply<2, 128>; using Streamed = TmaApply<2, 128>; using Recompute = TmaApply<2, 128, true>; };
template <> struct ApplyKernels<3> { using Affine = Affine2Apply<3, 64>;     using Streamed = TmaApply<3, 128>; using Recompute = TmaApply<3, 128, true>; };
template <> struct ApplyKernels<4> { using Affine = AffineApply<4, 64>;      using Streamed = TmaApply<4, 128>; using Recompute = TmaApply<4, 128, true>; };
template <> struct ApplyKernels<5> { using Affine = AffineApply<5, 64>;      using Streamed = TmaApply<5, 64>;  using Recompute = TmaApply<5, 64, true>; };
template <> struct ApplyKernels<6> { using Affine = MmaApply<6, MMA_AFFINE>; using Streamed = MmaApply<6, MMA_STREAMED>; using Recompute = MmaApply<6, MMA_RECOMPUTED>; };
template <> struct ApplyKernels<7> { using Affine = MmaApply<7, MMA_AFFINE>; using Streamed = MmaApply<7, MMA_STREAMED>; using Recompute = MmaApply<7, MMA_RECOMPUTED>; };
template <> struct ApplyKernels<8> { using Affine = ColumnApply<8>;          using Streamed = ColumnApply<8>;   using Recompute = ColumnApply<8, true>; };
// clang-format on

// Which entry of ApplyKernels<P> an operator runs
enum class ApplyGeometry
{
  Affine,
  Streamed,
  Recompute
};

// f(K{}) with K the launcher of the apply kernel of degree P for geometry mode `geo`
template <typename F>
void with_apply_kernel(int P, ApplyGeometry geo, F&& f)
{
  const auto pick = [&](auto deg)
  {
    using K = ApplyKernels<decltype(deg)::value>;
    if (geo == ApplyGeometry::Affine)
      f(typename K::Affine{});
    else if (geo == ApplyGeometry::Streamed)
      f(typename K::Streamed{});
    else
      f(typename K::Recompute{});
  };
  switch (P)
  {
  case 1: return pick(std::integral_constant<int, 1>{});
  case 2: return pick(std::integral_constant<int, 2>{});
  case 3: return pick(std::integral_constant<int, 3>{});
  case 4: return pick(std::integral_constant<int, 4>{});
  case 5: return pick(std::integral_constant<int, 5>{});
  case 6: return pick(std::integral_constant<int, 6>{});
  case 7: return pick(std::integral_constant<int, 7>{});
  case 8: return pick(std::integral_constant<int, 8>{});
  default:
    set_error("Unsupported degree");
    throw Error{PMGX_ERR_UNSUPPORTED};
  }
}

void upload_tables(pmgx_ctx* c)
{
  static double hD[PMGX_MAX_DEGREE + 1][MAXN * MAXN];
  static double hp[PMGX_MAX_DEGREE + 1][MAXN], hw[PMGX_MAX_DEGREE + 1][MAXN];
  std::memset(hD, 0, sizeof(hD));
  std::memset(hp, 0, sizeof(hp));
  std::memset(hw, 0, sizeof(hw));
  for (int P = 1; P <= PMGX_MAX_DEGREE; ++P)
  {
    std::vector<double> xs, ws, D;
    gll_points_weights(P + 1, xs, ws);
    gll_deriv_matrix(xs, D);
    for (int i = 0; i <= P; ++i)
      hp[P][i] = xs[i], hw[P][i] = ws[i];
    for (size_t i = 0; i < D.size(); ++i)
      hD[P][i] = D[i];
  }
  PMGX_CUDA(cudaMemcpyToSymbolAsync(c_D, hD, sizeof(hD), 0, cudaMemcpyHostToDevice, c->stream));
  PMGX_CUDA(cudaMemcpyToSymbolAsync(c_pts, hp, sizeof(hp), 0, cudaMemcpyHostToDevice, c->stream));
  PMGX_CUDA(cudaMemcpyToSymbolAsync(c_wts, hw, sizeof(hw), 0, cudaMemcpyHostToDevice, c->stream));
  PMGX_CUDA(cudaStreamSynchronize(c->stream));
}

inline int setup_grid(pmgx_ctx* c, long long total)
{
  long long b = (total + 255) / 256;
  long long cap = (long long)c->num_sms * 32;
  return (int)std::max<long long>(1, std::min(b, cap));
}
} // namespace

struct Laplacian : pmgx_operator
{
  int P = 0, n3 = 0;
  int n_cells = 0, n_l = 0, n_b = 0;
  const double* kappa = nullptr; // borrowed (cell_constants, src/laplacian.hpp:501)
  const int8_t* bc = nullptr;    // borrowed
  const double* xgeom = nullptr;
  const int32_t* geom_dofmap = nullptr;
  const int32_t* dofmap_borrowed = nullptr; // the caller's dofmap (borrowed like the reference's span, src/laplacian.hpp:502)
  int flags = 0;
  DevBuf<int32_t> perm; // launch position -> caller cell index (lcells then bcells)
  DevBuf<int32_t> enc;  // BC-encoded dofmap, layout `lay`
  DevBuf<double> G;     // geometry factors, layout `lay`
  Lay lay;
  DevBuf<double> Gc;   // [n_list][6] per-cell geometry factor of affine cells
  bool affine = false; // every cell affine: ApplyKernels<P>::Affine replaces the streamed-G kernel
  bool recompute = false; // PMGX_LAP_RECOMPUTE_G: no G, no Gc; every user of G forms it from xgeom
  bool q2 = false;        // PMGX_LAP_GEOM_Q2: 27 geometry nodes per cell

  int n_list() const { return n_l + n_b; }
  pmgx::ApplyGeometry geometry() const
  {
    return recompute ? pmgx::ApplyGeometry::Recompute
                     : (affine ? pmgx::ApplyGeometry::Affine : pmgx::ApplyGeometry::Streamed);
  }
  bool literal_detj() const { return (flags & PMGX_LAP_LITERAL_DETJ) != 0; }
  // G(p, comp, q) for the set-up kernels
  pmgx::StoredG stored_G() const { return {G.p, lay}; }
  pmgx::VertexG vertex_G() const { return {xgeom, geom_dofmap, perm.p, P, literal_detj()}; }

  void apply(double* x, double* y) override
  {
    cudaSetDevice(ctx->device);
    const long long ntot = (long long)n_owned + n_ghost;
    vec::set(ctx, y, ntot, 0.0); // out.set(0) :466 (fill kernel, see vec::set)
    if (halo)
      halo_fwd_begin(halo, x);                                                    // :378
    // interior cells on the compute stream; boundary + ghost cells right behind the exchange on
    // the halo stream: they start when the ghosts are in place and fill the interior kernel's tail
    // (both only add into y, which was zeroed before the exchange started).  Measured at 4 GPUs:
    // riding the halo stream wins at P1 (0.114 vs 0.121 ms), is neutral at P2 and loses 2 % at P4,
    // where the interior kernel is long enough to hide the join anyway
    const bool side = halo && P <= 2;
    cudaStream_t bs = side ? halo_stream(halo, ctx) : ctx->stream;
    const int lit = literal_detj();
    with_apply_kernel(P, geometry(), [&](auto k)
    {
      using K = decltype(k);
      const double* geom = K::cell_geometry ? Gc.p : G.p;
      K::launch(ctx, ctx->stream, {x, y, geom, enc.p, perm.p, kappa, 0, 0, n_l, xgeom, geom_dofmap, lit}); // :406-409
      if (halo && !side)
        halo_fwd_end(halo, x); // reference order: wait for the ghosts, then the boundary launch (:425)
      K::launch(ctx, bs, {x, y, geom, enc.p, perm.p, kappa, lay.nb_l, n_l, n_b, xgeom, geom_dofmap, lit}); // :449-452
    });
    if (side)
      halo_fwd_end(halo, x);                                                      // :425 (join)
  }
};
} // namespace pmgx

using pmgx::Laplacian;

extern "C"
{
int pmgx_laplacian_create(pmgx_ctx* ctx, int degree, int n_cells, const int32_t* dofmap,
                          const double* xgeom, int n_points, const int32_t* geom_dofmap,
                          const double* kappa, const int32_t* lcells_h, int n_lcells,
                          const int32_t* bcells_h, int n_bcells, const int8_t* bc_marker,
                          int n_owned, int n_ghost, pmgx_halo* halo, int flags, pmgx_operator** out)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(ctx && out, "laplacian_create: null ctx/out");
  if (degree < 1 || degree > PMGX_MAX_DEGREE)
  {
    pmgx::set_error("Unsupported degree"); // same message as src/laplacian.hpp:346,479
    return PMGX_ERR_UNSUPPORTED;
  }
  PMGX_REQUIRE(n_cells >= 0 && n_lcells >= 0 && n_bcells >= 0 && n_lcells + n_bcells <= n_cells,
               "laplacian_create: inconsistent cell counts");
  PMGX_REQUIRE(n_cells == 0 || (dofmap && xgeom && geom_dofmap && kappa && bc_marker),
               "laplacian_create: null array");
  PMGX_REQUIRE(n_owned >= 0 && n_ghost >= 0 && n_points >= 0, "laplacian_create: bad sizes");
  PMGX_REQUIRE(!halo || (halo->n_owned == n_owned && halo->n_ghost == n_ghost),
               "laplacian_create: halo does not match the vector layout");
  if ((flags & PMGX_LAP_GEOM_Q2) && (flags & PMGX_LAP_RECOMPUTE_G))
  {
    pmgx::set_error("laplacian_create: PMGX_LAP_GEOM_Q2 is not supported with PMGX_LAP_RECOMPUTE_G (the recompute "
                    "apply kernels form trilinear Jacobians only)");
    return PMGX_ERR_UNSUPPORTED;
  }
  PMGX_CUDA(cudaSetDevice(ctx->device));
  pmgx::upload_tables(ctx);

  auto* L = new Laplacian();
  std::unique_ptr<Laplacian> guard(L);
  L->ctx = ctx;
  L->kind = pmgx_operator::LAPLACIAN;
  L->P = degree;
  const int n = degree + 1;
  L->n3 = n * n * n;
  L->n_cells = n_cells;
  L->n_l = n_lcells;
  L->n_b = n_bcells;
  L->n_owned = n_owned;
  L->n_ghost = n_ghost;
  L->halo = halo;
  L->kappa = kappa;
  L->bc = bc_marker;
  L->xgeom = xgeom;
  L->geom_dofmap = geom_dofmap;
  L->dofmap_borrowed = dofmap;
  L->flags = flags;
  L->recompute = (flags & PMGX_LAP_RECOMPUTE_G) != 0;
  L->q2 = (flags & PMGX_LAP_GEOM_Q2) != 0;

  const int n_list = L->n_list();
  std::vector<int32_t> perm_h((size_t)n_list);
  for (int i = 0; i < n_lcells; ++i)
    perm_h[i] = lcells_h[i];
  for (int i = 0; i < n_bcells; ++i)
    perm_h[n_lcells + i] = bcells_h[i];
  for (int32_t v : perm_h)
    PMGX_REQUIRE(v >= 0 && v < n_cells, "laplacian_create: cell index %d out of range", v);
  L->perm.upload(perm_h.data(), perm_h.size(), ctx->stream);

  const long long total = (long long)n_list * L->n3;
  pmgx::Lay& lay = L->lay;
  lay.n = n, lay.n2 = n * n, lay.n3 = L->n3;
  lay.n_l = n_lcells;
  // affine cells: one geometry 6-vector per cell instead of one per quadrature point, for the degrees
  // that have a kernel for it (decided first: the layout follows the kernel that will run)
  bool has_affine_kernel = false;
  pmgx::with_apply_kernel(degree, pmgx::ApplyGeometry::Affine,
                          [&](auto k) { has_affine_kernel = decltype(k)::cell_geometry; });
  if (n_list > 0 && has_affine_kernel && !(flags & PMGX_LAP_STREAM_G) && !L->recompute)
  {
    L->Gc.alloc((size_t)n_list * 6);
    pmgx::DevBuf<int> bad;
    bad.alloc(1);
    PMGX_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(int), ctx->stream));
    if (L->q2)
      pmgx::k_cell_geometry_q2<<<(n_list + 255) / 256, 256, 0, ctx->stream>>>(
          xgeom, geom_dofmap, L->perm.p, L->Gc.p, n_list, (flags & PMGX_LAP_LITERAL_DETJ) != 0, 1e-13, bad.p);
    else
      pmgx::k_cell_geometry<<<(n_list + 255) / 256, 256, 0, ctx->stream>>>(
          xgeom, geom_dofmap, L->perm.p, L->Gc.p, n_list, (flags & PMGX_LAP_LITERAL_DETJ) != 0, 1e-13, bad.p);
    pmgx::check_launch("k_cell_geometry");
    pmgx::count_launch(ctx);
    int n_bad = 0;
    PMGX_CUDA(cudaMemcpyAsync(&n_bad, bad.p, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    PMGX_CUDA(cudaStreamSynchronize(ctx->stream));
    L->affine = n_bad == 0;
    if (!L->affine)
      L->Gc.release();
  }
  pmgx::with_apply_kernel(degree, L->geometry(), [&](auto k) { lay.cpb = decltype(k)::cpb; });
  lay.mode = lay.cpb > 0 ? 1 : 0;
  if (lay.mode == 1)
  {
    lay.S = (lay.cpb * n + 1) & ~1;
    lay.SE = (lay.cpb * n + 3) & ~3;
    lay.nb_l = (n_lcells + lay.cpb - 1) / lay.cpb;
    lay.n_batches = lay.nb_l + (n_bcells + lay.cpb - 1) / lay.cpb;
  }
  const long long enc_size = lay.mode == 1 ? lay.enc_size() : total;
  const long long g_size = L->recompute ? 0 : (lay.mode == 1 ? lay.g_size() : total * 6);
  L->enc.alloc((size_t)enc_size);
  L->G.alloc((size_t)g_size);
  if (lay.mode == 1 && enc_size > 0)
  { // padded slots: inert
    PMGX_CUDA(cudaMemsetAsync(L->enc.p, 0, (size_t)enc_size * sizeof(int32_t), ctx->stream));
    if (g_size > 0)
      PMGX_CUDA(cudaMemsetAsync(L->G.p, 0, (size_t)g_size * sizeof(double), ctx->stream));
  }
  if (total > 0)
  {
    pmgx::k_encode_dofmap<<<pmgx::setup_grid(ctx, total), 256, 0, ctx->stream>>>(
        dofmap, L->perm.p, bc_marker, L->enc.p, L->n3, total, lay);
    pmgx::check_launch("k_encode_dofmap");
    pmgx::count_launch(ctx);
    if (L->q2)
    {
      pmgx::k_geometry_q2<true><<<pmgx::setup_grid(ctx, 32ll * n_list), 32 * pmgx::Q2_GEOM_WARPS, 0, ctx->stream>>>(
          degree, xgeom, geom_dofmap, L->perm.p, L->G.p, nullptr, n_list, (flags & PMGX_LAP_LITERAL_DETJ) != 0, lay);
      pmgx::check_launch("k_geometry_q2");
      pmgx::count_launch(ctx);
    }
    else if (!L->recompute)
    {
      pmgx::k_geometry<true><<<pmgx::setup_grid(ctx, total), 256, 0, ctx->stream>>>(
          degree, xgeom, geom_dofmap, L->perm.p, L->G.p, nullptr, n_list,
          (flags & PMGX_LAP_LITERAL_DETJ) != 0, lay);
      pmgx::check_launch("k_geometry");
      pmgx::count_launch(ctx);
    }
  }
  L->diag_inv.alloc((size_t)n_owned);
  if (!(flags & PMGX_LAP_NO_DIAG) && n_owned > 0)
  {
    pmgx::DevBuf<double> diag;
    diag.alloc((size_t)n_owned + n_ghost);
    PMGX_CUDA(cudaMemsetAsync(diag.p, 0, diag.n * sizeof(double), ctx->stream));
    if (total > 0)
    {
      if (L->recompute)
        pmgx::k_diag<<<pmgx::setup_grid(ctx, total), 256, 0, ctx->stream>>>(
            degree, L->vertex_G(), L->enc.p, L->perm.p, kappa, diag.p, n_list, lay);
      else
        pmgx::k_diag<<<pmgx::setup_grid(ctx, total), 256, 0, ctx->stream>>>(
            degree, L->stored_G(), L->enc.p, L->perm.p, kappa, diag.p, n_list, lay);
      pmgx::check_launch("k_diag");
    }
    pmgx::k_invert_diag<<<(n_owned + 255) / 256, 256, 0, ctx->stream>>>(diag.p, bc_marker,
                                                                         L->diag_inv.p, n_owned);
    pmgx::check_launch("k_invert_diag");
    pmgx::count_launch(ctx, 2);
    PMGX_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  else if (n_owned > 0)
    PMGX_CUDA(cudaMemsetAsync(L->diag_inv.p, 0, (size_t)n_owned * sizeof(double), ctx->stream));
  PMGX_CUDA(cudaStreamSynchronize(ctx->stream));
  *out = guard.release();
  PMGX_API_END
}

int pmgx_laplacian_get_G(pmgx_operator* op, double* G_out)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(op && op->kind == pmgx_operator::LAPLACIAN && G_out, "laplacian_get_G: bad arguments");
  auto* L = static_cast<Laplacian*>(op);
  const long long total = (long long)L->n_list() * L->n3 * 6;
  if (total > 0)
  {
    PMGX_CUDA(cudaSetDevice(L->ctx->device));
    if (L->recompute) // straight into the caller's buffer: no G exists
      pmgx::k_G_to_reference_layout<<<pmgx::setup_grid(L->ctx, total), 256, 0, L->ctx->stream>>>(
          L->vertex_G(), G_out, L->n3, total);
    else
      pmgx::k_G_to_reference_layout<<<pmgx::setup_grid(L->ctx, total), 256, 0, L->ctx->stream>>>(
          L->stored_G(), G_out, L->n3, total);
    pmgx::check_launch("k_G_to_reference_layout");
    pmgx::count_launch(L->ctx);
  }
  PMGX_API_END
}

int pmgx_laplacian_is_affine(pmgx_operator* op)
{
  return op && op->kind == pmgx_operator::LAPLACIAN && static_cast<Laplacian*>(op)->affine ? 1 : 0;
}

int pmgx_laplacian_kernel_name(pmgx_operator* op, char* name_h, int cap)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(op && op->kind == pmgx_operator::LAPLACIAN && name_h && cap > 0, "laplacian_kernel_name: bad arguments");
  auto* L = static_cast<Laplacian*>(op);
  pmgx::with_apply_kernel(L->P, L->geometry(), [&](auto k) { decltype(k)::name(name_h, cap); });
  PMGX_API_END
}

int pmgx_laplacian_device_bytes(pmgx_operator* op, long long* bytes_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(op && op->kind == pmgx_operator::LAPLACIAN && bytes_h, "laplacian_device_bytes: bad arguments");
  auto* L = static_cast<Laplacian*>(op);
  *bytes_h = (long long)(L->perm.n * sizeof(int32_t) + L->enc.n * sizeof(int32_t) + L->G.n * sizeof(double)
                         + L->Gc.n * sizeof(double) + L->diag_inv.n * sizeof(double));
  PMGX_API_END
}

int pmgx_laplacian_rhs(pmgx_operator* op, const double* fvals, double g, double* b)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(op && op->kind == pmgx_operator::LAPLACIAN && fvals && b, "laplacian_rhs: bad arguments");
  auto* L = static_cast<Laplacian*>(op);
  pmgx_ctx* ctx = L->ctx;
  PMGX_CUDA(cudaSetDevice(ctx->device));
  const long long total = (long long)L->n_list() * L->n3;
  const int ntot = L->n_owned + L->n_ghost;
  PMGX_CUDA(cudaMemsetAsync(b, 0, (size_t)ntot * sizeof(double), ctx->stream));
  if (total > 0)
  {
    pmgx::DevBuf<double> dw;
    dw.alloc((size_t)total);
    if (L->q2)
      pmgx::k_geometry_q2<false><<<pmgx::setup_grid(ctx, 32ll * L->n_list()), 32 * pmgx::Q2_GEOM_WARPS, 0, ctx->stream>>>(
          L->P, L->xgeom, L->geom_dofmap, L->perm.p, nullptr, dw.p, L->n_list(), false, L->lay);
    else
      pmgx::k_geometry<false><<<pmgx::setup_grid(ctx, total), 256, 0, ctx->stream>>>(
          L->P, L->xgeom, L->geom_dofmap, L->perm.p, nullptr, dw.p, L->n_list(), false, L->lay);
    pmgx::check_launch("k_geometry(detJ)");
    pmgx::k_rhs<<<pmgx::setup_grid(ctx, total), 256, 0, ctx->stream>>>(dw.p, L->enc.p, fvals, b, total, L->n3, L->lay);
    pmgx::check_launch("k_rhs");
    pmgx::count_launch(ctx, 2);
    PMGX_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  if (ntot > 0 && g != 0.0)
  {
    // inhomogeneous data: b -= A_full g_bc, then set_bc (examples/pmg/main.cpp:293-295)
    pmgx::DevBuf<double> gv;
    gv.alloc((size_t)ntot);
    pmgx::k_fill<<<(ntot + 255) / 256, 256, 0, ctx->stream>>>(gv.p, g, ntot);
    pmgx::check_launch("k_fill");
    const int rc = pmgx_laplacian_lift(op, gv.p, b);
    if (rc != PMGX_OK)
      return rc;
    PMGX_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  else if (ntot > 0)
  {
    pmgx::k_set_bc_value<<<(ntot + 255) / 256, 256, 0, ctx->stream>>>(b, L->bc, g, ntot);
    pmgx::check_launch("k_set_bc_value");
    pmgx::count_launch(ctx);
  }
  PMGX_API_END
}

int pmgx_laplacian_lift(pmgx_operator* op, const double* gvals, double* b)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(op && op->kind == pmgx_operator::LAPLACIAN && gvals && b, "laplacian_lift: bad arguments");
  auto* L = static_cast<Laplacian*>(op);
  pmgx_ctx* ctx = L->ctx;
  PMGX_CUDA(cudaSetDevice(ctx->device));
  const int ntot = L->n_owned + L->n_ghost;
  if (ntot == 0)
    return PMGX_OK;
  // the same cells, geometry and kappa with an all-zero Dirichlet marker: A_full.  No halo: g_bc is
  // given on owned AND ghost dofs, and the ghost cells make the owned rows complete.
  pmgx::DevBuf<int8_t> nobc;
  nobc.alloc((size_t)ntot);
  PMGX_CUDA(cudaMemsetAsync(nobc.p, 0, (size_t)ntot, ctx->stream));
  std::vector<int32_t> perm_h((size_t)L->n_list());
  if (!perm_h.empty())
    PMGX_CUDA(cudaMemcpy(perm_h.data(), L->perm.p, perm_h.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
  pmgx_operator* full = nullptr;
  const int n_points_unknown = 0; // only used for argument checks
  const int rc = pmgx_laplacian_create(ctx, L->P, L->n_cells, L->dofmap_borrowed, L->xgeom, n_points_unknown, L->geom_dofmap,
                                       L->kappa, perm_h.data(), (int)perm_h.size(), nullptr, 0, nobc.p, L->n_owned,
                                       L->n_ghost, nullptr,
                                       (L->flags & (PMGX_LAP_LITERAL_DETJ | PMGX_LAP_RECOMPUTE_G | PMGX_LAP_GEOM_Q2)) | PMGX_LAP_NO_DIAG,
                                       &full);
  if (rc != PMGX_OK)
    return rc;
  pmgx::DevBuf<double> gbc, y;
  gbc.alloc((size_t)ntot);
  y.alloc((size_t)ntot);
  pmgx::k_mask_to_bc<<<(ntot + 255) / 256, 256, 0, ctx->stream>>>(gvals, L->bc, gbc.p, ntot);
  pmgx::check_launch("k_mask_to_bc");
  full->apply(gbc.p, y.p);
  pmgx::k_lift<<<(L->n_owned + 255) / 256, 256, 0, ctx->stream>>>(b, y.p, gvals, L->bc, L->n_owned);
  pmgx::check_launch("k_lift");
  pmgx::count_launch(ctx, 2);
  PMGX_CUDA(cudaStreamSynchronize(ctx->stream));
  pmgx_operator_destroy(full);
  PMGX_API_END
}

int pmgx_csr_from_laplacian(pmgx_operator* op, pmgx_operator** out)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(op && op->kind == pmgx_operator::LAPLACIAN && out, "csr_from_laplacian: bad arguments");
  auto* L = static_cast<Laplacian*>(op);
  pmgx_ctx* ctx = L->ctx;
  PMGX_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int n_owned = L->n_owned;
  const long long ntot = (long long)L->n_owned + L->n_ghost;
  const long long n_list = L->n_list();
  const long long per_cell = (long long)L->n3 * L->n3;
  const long long n_trip = n_list * per_cell + n_owned;
  pmgx::DevBuf<unsigned long long> keys, ukeys;
  pmgx::DevBuf<double> vals, uvals;
  keys.alloc((size_t)std::max<long long>(n_trip, 1));
  vals.alloc((size_t)std::max<long long>(n_trip, 1));
  if (n_list > 0)
  {
    if (L->recompute)
      pmgx::k_element_triplets<<<pmgx::setup_grid(ctx, n_list * per_cell), 256, 0, st>>>(
          L->P, L->vertex_G(), L->enc.p, L->perm.p, L->kappa, n_list, n_owned, ntot, keys.p, vals.p, L->lay);
    else
      pmgx::k_element_triplets<<<pmgx::setup_grid(ctx, n_list * per_cell), 256, 0, st>>>(
          L->P, L->stored_G(), L->enc.p, L->perm.p, L->kappa, n_list, n_owned, ntot, keys.p, vals.p, L->lay);
    pmgx::check_launch("k_element_triplets");
  }
  if (n_owned > 0)
  {
    pmgx::k_bc_diag_triplets<<<(n_owned + 255) / 256, 256, 0, st>>>(
        L->bc, n_owned, ntot, keys.p + n_list * per_cell, vals.p + n_list * per_cell);
    pmgx::check_launch("k_bc_diag_triplets");
  }
  auto pol = thrust::cuda::par.on(st);
  thrust::device_ptr<unsigned long long> kp(keys.p);
  thrust::device_ptr<double> vp(vals.p);
  thrust::stable_sort_by_key(pol, kp, kp + n_trip, vp);
  ukeys.alloc((size_t)std::max<long long>(n_trip, 1));
  uvals.alloc((size_t)std::max<long long>(n_trip, 1));
  thrust::device_ptr<unsigned long long> ukp(ukeys.p);
  thrust::device_ptr<double> uvp(uvals.p);
  auto ends = thrust::reduce_by_key(pol, kp, kp + n_trip, vp, ukp, uvp);
  long long nnz = ends.first - ukp;
  if (nnz > 0)
  {
    unsigned long long last;
    PMGX_CUDA(cudaMemcpyAsync(&last, ukeys.p + nnz - 1, sizeof(last), cudaMemcpyDeviceToHost, st));
    PMGX_CUDA(cudaStreamSynchronize(st));
    if (last == ~0ull)
      --nnz; // the sentinel group sorts last
  }
  PMGX_REQUIRE(nnz < (1ll << 31), "csr_from_laplacian: more than 2^31 non-zeros");
  keys.release();
  vals.release();

  std::unique_ptr<pmgx::CsrOperator> A(new pmgx::CsrOperator());
  A->ctx = ctx;
  A->kind = pmgx_operator::CSR;
  A->n_owned = n_owned;
  A->n_ghost = L->n_ghost;
  A->halo = L->halo;
  A->nnz = nnz;
  A->row_ptr.alloc((size_t)n_owned + 1);
  A->off_diag.alloc((size_t)n_owned);
  A->cols.alloc((size_t)std::max<long long>(nnz, 1));
  A->values.alloc((size_t)std::max<long long>(nnz, 1));
  pmgx::DevBuf<int32_t> row_count, owned_count;
  row_count.alloc((size_t)n_owned + 1);
  owned_count.alloc((size_t)n_owned + 1);
  PMGX_CUDA(cudaMemsetAsync(row_count.p, 0, ((size_t)n_owned + 1) * sizeof(int32_t), st));
  PMGX_CUDA(cudaMemsetAsync(owned_count.p, 0, ((size_t)n_owned + 1) * sizeof(int32_t), st));
  if (nnz > 0)
  {
    pmgx::k_split_keys<<<pmgx::setup_grid(ctx, nnz), 256, 0, st>>>(ukeys.p, nnz, ntot, n_owned, A->cols.p,
                                                                 row_count.p, owned_count.p);
    pmgx::check_launch("k_split_keys");
    PMGX_CUDA(cudaMemcpyAsync(A->values.p, uvals.p, (size_t)nnz * sizeof(double), cudaMemcpyDeviceToDevice, st));
  }
  thrust::device_ptr<int32_t> rc(row_count.p), rp(A->row_ptr.p);
  thrust::exclusive_scan(pol, rc, rc + n_owned + 1, rp);
  if (n_owned > 0)
  {
    pmgx::k_offdiag<<<(n_owned + 255) / 256, 256, 0, st>>>(A->row_ptr.p, owned_count.p, n_owned, A->off_diag.p);
    pmgx::check_launch("k_offdiag");
  }
  pmgx::count_launch(ctx, 6);
  PMGX_CUDA(cudaStreamSynchronize(st));
  // does any row address ghost columns?
  {
    thrust::device_ptr<int32_t> oc(owned_count.p);
    const long long owned_total = thrust::reduce(pol, oc, oc + n_owned, (long long)0);
    A->has_ghost_cols = owned_total < nnz;
  }
  A->finish_setup();
  *out = A.release();
  PMGX_API_END
}

// ----------------------------------------------------------------- generic operator --
int pmgx_operator_apply(pmgx_operator* op, double* x, double* y)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(op && x && y, "operator_apply: null argument");
  PMGX_REQUIRE(x != y, "operator_apply: in-place apply is not supported");
  op->apply(x, y);
  PMGX_API_END
}

int pmgx_operator_get_diag_inverse(pmgx_operator* op, double* out)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(op && out, "get_diag_inverse: null argument");
  pmgx::vec::copy(op->ctx, out, op->diag_inv.p, op->n_owned);
  PMGX_API_END
}

int pmgx_operator_set_diag_inverse(pmgx_operator* op, const double* in)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(op && in, "set_diag_inverse: null argument");
  pmgx::vec::copy(op->ctx, op->diag_inv.p, in, op->n_owned);
  PMGX_API_END
}

int pmgx_operator_n_owned(pmgx_operator* op) { return op ? op->n_owned : -1; }
int pmgx_operator_n_ghost(pmgx_operator* op) { return op ? op->n_ghost : -1; }

int pmgx_operator_destroy(pmgx_operator* op)
{
  PMGX_API_BEGIN
  if (op)
  {
    cudaSetDevice(op->ctx->device);
    cudaStreamSynchronize(op->ctx->stream);
    delete op;
  }
  PMGX_API_END
}
}
