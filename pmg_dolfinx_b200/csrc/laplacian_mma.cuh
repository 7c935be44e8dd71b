// FP64 tensor-core (DMMA, mma.sync.m8n8k4.f64) apply kernel for HIGH degree on affine cells: P6 and P7
// (n = P + 1 = 7, 8 points per direction, padded to the 8-wide tile).  Included by laplacian.cu inside
// namespace pmgx::{anonymous} (it uses the constant tables c_D / c_wts defined there).
//
// Why a different mapping at high degree (north_star item 1; DESIGN.md section 3.1): the slab kernels keep
// 2 n^2 doubles of an element per thread -- 255 registers and spills at n >= 7, two warps per scheduler,
// 8 TFLOP/s.  With DMMA the element lives in shared memory and its fragments are spread over a WARP, and at
// n = 7, 8 the 8x8x4 tiles are 77-100 % full.  The FP64 rate itself is the same as the FMA pipe's (measured:
// 37 vs 34 TFLOP/s, one datapath) -- the gain is the register relief, not the pipe.  Below P5 the tiles
// would be <= 40 % full: the slab kernels stay.
//
// One WARP per cell.  Two lane layouts of the 8x8x8 points, both the accumulator layout of the mma:
//   Y: lane (r = lane/4, c = lane%4) holds the points (i = t, j = r, k = 2c + {0,1}), t = 0..7
//   X: ...                                 the points (i = r, j = t, k = 2c + {0,1})
// Per cell:
//   gather   dof indices and u in layout Y (for n = 8 that is the linear order: one 8-byte index load per t)
//   forward  for every tile t: gz(t,.,.) = U[t] D^T   (A = U[t][j][m] from smem, B = D^T in registers)   -> Y
//                              gy(t,.,.) = D U[t]     (A = D in registers,  B = U[t][m][k] from smem)    -> Y
//                              gx(.,t,.) = D U[.][t]  (A = D in registers,  B = U[m][t][k] from smem)    -> X
//   re-layout gx X -> Y through shared memory (16-byte stores / loads), flux (fx, fy, fz) = w Gc grad in
//            registers at the Y points, stored once (16-byte stores)
//   backward the transposed contractions: fz and fy into one accumulator (Y), fx into another (X)
//   combine  the X accumulator goes through shared memory to Y; every lane scatters its Y points (atomics)
// Shared memory per warp: three 8x8x8 arrays, i-stride 72, j-stride 8 doubles, k XOR-swizzled with
// 4 ((i/2 + j/2) mod 2): every access pattern above -- 8-byte fragment loads over (4 x 4) blocks of (j,k) or
// (i,k), 16-byte accumulator accesses over (2 x 8) blocks -- is bank-conflict free.  The first version
// (padded strides 100 / 12, fluxes accumulated in shared memory in two passes) ran at 71 % of the shared-memory
// wavefront peak with 41 % of the wavefronts being conflicts (profiles/r2_apply_p7_mma.txt); this data flow
// needs 2.5x fewer wavefronts.  tests/test_mma_emulation.py runs the same lane-level index logic in numpy
// against the oracle and counts the bank conflicts of every access.
#pragma once

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b)
{
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

template <int P, int WPB>
struct MmaCfg
{
  static constexpr int n = P + 1;
  static constexpr int n3 = n * n * n;
  static constexpr int SI = 72;       // i-stride (doubles); j-stride 8; k swizzled, see at()
  static constexpr int arr = 8 * SI;  // doubles per array
  static constexpr size_t smem = (size_t)WPB * 3 * arr * sizeof(double);
  __host__ __device__ static constexpr int at(int i, int j, int k)
  {
    return i * SI + j * 8 + (k ^ ((((i >> 1) ^ (j >> 1)) & 1) << 2));
  }
};

// Where the kernel takes the geometry from:
//   MMA_AFFINE    : Gc[p][6], one geometry 6-vector per (affine) cell, quadrature weights applied here;
//   MMA_STREAMED  : Gc = G[p][6][n3], the reference's data flow (G per quadrature point, weights folded in),
//                   read in layout Y one tile ahead of the flux that uses it; at P6 the cell's whole block is
//                   prefetched into L2 first;
//   MMA_RECOMPUTED: no G; the cell's 8 vertices go to 24 doubles of per-warp shared memory beside the three
//                   arrays, and every lane forms G at its two points of tile t from its JacobianAlongXi pair
//                   (fixed eta_r, zeta_{2c+h}) right where the streamed variant consumes its G registers.
enum MmaGeometry
{
  MMA_AFFINE,
  MMA_STREAMED,
  MMA_RECOMPUTED
};
template <int P, int WPB, int MINB, int GEO>
__global__ void __launch_bounds__(WPB * 32, MINB)
k_apply_affine_mma(const double* __restrict__ x, double* __restrict__ y, const double* __restrict__ Gc,
                   const int32_t* __restrict__ enc, const int32_t* __restrict__ perm,
                   const double* __restrict__ kappa, int first, int count, const double* __restrict__ xgeom,
                   const int32_t* __restrict__ geom_dofmap, int literal_detj)
{
  using C = MmaCfg<P, WPB>;
  constexpr int n = C::n, n3 = C::n3, SI = C::SI;
  constexpr bool STREAM = GEO == MMA_STREAMED, RECOMPUTE = GEO == MMA_RECOMPUTED;
  extern __shared__ __align__(16) double smem_mma[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double* const B0 = smem_mma + (size_t)warp * 3 * C::arr; // U, then gx in transit, then fx
  double* const B1 = B0 + C::arr;                          // fy, then the X accumulator in transit
  double* const B2 = B1 + C::arr;                          // fz
  double* const SV = smem_mma + (size_t)WPB * 3 * C::arr + warp * 24; // RECOMPUTE: the cell's vertices [8][3]
  for (int i = lane; i < 3 * C::arr; i += 32)
    B0[i] = 0.0; // planes i >= n are never written again: everything the tiles read there is an exact zero
  __syncwarp();

  const int r = lane >> 2, c = lane & 3;
  const int sr = (r >> 1) & 1, sc = (c >> 1) & 1;
  // lane parts of the swizzled addresses, indexed by the swizzle bit of the unrolled (compile-time) index t
  const int yo[2] = {r * 8 + ((2 * c) ^ (4 * sr)), r * 8 + ((2 * c) ^ (4 * (sr ^ 1)))};     // (t, r, 2c): + t SI
  const int xo[2] = {r * SI + ((2 * c) ^ (4 * sr)), r * SI + ((2 * c) ^ (4 * (sr ^ 1)))};   // (r, t, 2c): + 8 t
  const int f1[2] = {r * 8 + (c ^ (4 * sr)), r * 8 + (c ^ (4 * (sr ^ 1)))};                 // (t, r, c): + t SI
  const int f2[2] = {c * 8 + (r ^ (4 * sc)), c * 8 + (r ^ (4 * (sc ^ 1)))};                 // (t, c, r): + t SI
  const int f3[2] = {c * SI + (r ^ (4 * sc)), c * SI + (r ^ (4 * (sc ^ 1)))};               // (c, t, r): + 8 t
  auto Dp = [&](int a, int b) -> double { return (a < n && b < n) ? c_D[P][a * n + b] : 0.0; };
  auto Wp = [&](int a) -> double { return a < n ? c_wts[P][a] : 0.0; };
  // fragments of the derivative table: A = D (also B = D^T: the same values), A = D^T (also B = D)
  const double dA0 = Dp(r, c), dA1 = Dp(r, c + 4);
  const double tA0 = Dp(c, r), tA1 = Dp(c + 4, r);
  const double wr0 = Wp(r) * Wp(2 * c), wr1 = Wp(r) * Wp(2 * c + 1);
  const bool v0 = r < n && 2 * c < n, v1 = r < n && 2 * c + 1 < n; // the lane's two points exist (n = 7 pads)

  const int gw = blockIdx.x * WPB + warp, nw = gridDim.x * WPB;
  // this lane's dof indices of cell pl (layout Y), -1 where the lane has no point
  auto load_idx = [&](int pl, int32_t (*d)[2])
  {
    const int32_t* e = enc + ((long long)first + pl) * n3;
#pragma unroll
    for (int t = 0; t < n; ++t)
    {
      if constexpr (n == 8)
      {
        const int2 dd = __ldcs(reinterpret_cast<const int2*>(e + 64 * t) + lane);
        d[t][0] = dd.x;
        d[t][1] = dd.y;
      }
      else
      {
        const int a = t * n * n + r * n + 2 * c;
        d[t][0] = v0 ? ldg_stream_i32(e + a) : -1;
        d[t][1] = v1 ? ldg_stream_i32(e + a + 1) : -1;
      }
    }
  };
  // STREAM: the indices are loaded one cell ahead (before the transposed contractions, when the forward
  // accumulators are dead), so one global round trip of the gather is exposed per cell instead of two.  Measured
  // at 100 M dofs, ahead vs not: streamed P6 2.13 vs 2.22 ms, P7 1.74 vs 1.76 ms; affine P6 1.55 vs 1.42 ms,
  // P7 1.21 vs 1.20 ms (there the 16 extra live registers cost more than the round trip: 88 bytes of spills)
  constexpr bool AHEAD = STREAM;
  int32_t d[n][2], dn[n][2];
  if (AHEAD && gw < count)
    load_idx(gw, d);
  for (int pl = gw; pl < count; pl += nw)
  {
    const long long p = (long long)first + pl;
    double xv[n][2];
    if constexpr (!AHEAD)
      load_idx(pl, d);
    // gather (Dirichlet columns zeroed: src/laplacian.hpp:186-187): all index loads in one sweep (above, or one
    // cell ahead), all value loads in the next.  No global store may sit between the loads: with the
    // Dirichlet-row stores y = x in this loop (as in the slab kernels) every index -> value -> store chain was
    // exposed at full latency, even with the store predicated off (ncu: long_scoreboard 28.7 stalls per issue,
    // 4.4 ms instead of 1.2 ms at P7); they are done in the scatter, under a branch.
#pragma unroll
    for (int t = 0; t < n; ++t)
#pragma unroll
      for (int h = 0; h < 2; ++h)
        xv[t][h] = d[t][h] >= 0 ? x[d[t][h]] : 0.0;
#pragma unroll
    for (int t = 0; t < n; ++t)
      *reinterpret_cast<double2*>(B0 + t * SI + yo[(t >> 1) & 1]) = make_double2(xv[t][0], xv[t][1]);
    const double kap = kappa[perm[p]]; // re-read on every apply (src/laplacian.hpp:230)
    if constexpr (RECOMPUTE)
    { // the previous cell's reads of SV ended before the barrier after its flux phase
      if (lane < 24)
        SV[lane] = xgeom[3ll * geom_dofmap[(long long)perm[p] * 8 + lane / 3] + lane % 3];
    }
    double G00 = 0, G01 = 0, G02 = 0, G11 = 0, G12 = 0, G22 = 0;
    const double* Gq = nullptr; // STREAM: this lane's first point of the cell's G block
    double2 gq[2][6];           // STREAM: G of the lane's two points, tiles t (flux) and t + 1 (in flight)
    auto load_g = [&](int t, double2* g)
    {
#pragma unroll
      for (int cc = 0; cc < 6; ++cc)
      {
        if constexpr (n == 8)
          g[cc] = __ldcs(reinterpret_cast<const double2*>(Gq + cc * n3 + 64 * t));
        else
        {
          const double* q = Gq + cc * n3 + t * n * n;
          g[cc] = make_double2(v0 ? ldg_stream(q) : 0.0, v1 ? ldg_stream(q + 1) : 0.0);
        }
      }
    };
    if constexpr (STREAM)
    {
      Gq = Gc + (size_t)p * 6 * n3 + (n == 8 ? 2 * lane : r * n + 2 * c);
      // L2 prefetch of this cell's G block, measured at 100 M dofs (none / this cell / next cell): P6 2.36 / 2.22 /
      // 2.23 ms, P7 1.76 / 1.85 / 2.19 ms (at n = 8 the 16-byte tile loads stream well on their own and the prefetch
      // only adds DRAM traffic: 12.3 GB against 9.3 GB algorithmic, profiles/r2_apply_p7_mma.txt)
      if constexpr (P == 6)
      { // 6 n3 doubles, 128-byte lines
        const uintptr_t b0 = reinterpret_cast<uintptr_t>(Gc + (size_t)p * 6 * n3), b1 = b0 + 6 * n3 * 8;
        for (uintptr_t a = (b0 & ~(uintptr_t)127) + 128 * lane; a < b1; a += 128 * 32)
          asm volatile("prefetch.global.L2 [%0];" ::"l"(a));
      }
      load_g(0, gq[0]);
    }
    else if constexpr (GEO == MMA_AFFINE)
    {
      const double* gp = Gc + (size_t)p * 6;
      G00 = gp[0] * kap, G01 = gp[1] * kap, G02 = gp[2] * kap, G11 = gp[3] * kap, G12 = gp[4] * kap, G22 = gp[5] * kap;
    }
    __syncwarp();
    // ---- forward contractions
    double gz[n][2], gy[n][2], gx[n][2];
#pragma unroll
    for (int t = 0; t < n; ++t)
    {
      const int b = (t >> 1) & 1;
      gz[t][0] = gz[t][1] = gy[t][0] = gy[t][1] = gx[t][0] = gx[t][1] = 0.0;
      dmma884(gz[t][0], gz[t][1], B0[t * SI + f1[b]], dA0);            // k = c     (f1[b] ^ 4 is k = c + 4)
      dmma884(gz[t][0], gz[t][1], B0[t * SI + (f1[b] ^ 4)], dA1);
      dmma884(gy[t][0], gy[t][1], dA0, B0[t * SI + f2[b]]);            // j = c, then j = c + 4
      dmma884(gy[t][0], gy[t][1], dA1, B0[t * SI + 32 + f2[b]]);
      dmma884(gx[t][0], gx[t][1], dA0, B0[t * 8 + f3[b]]);             // i = c, then i = c + 4
      dmma884(gx[t][0], gx[t][1], dA1, B0[t * 8 + 4 * SI + f3[b]]);
    }
    __syncwarp(); // every lane is done reading U: B0 carries gx from layout X to layout Y
#pragma unroll
    for (int t = 0; t < n; ++t)
      *reinterpret_cast<double2*>(B0 + t * 8 + xo[(t >> 1) & 1]) = make_double2(gx[t][0], gx[t][1]);
    __syncwarp();
    // ---- flux at the Y points (i = t, j = r, k = 2c + h); a lane overwrites only the slots it has just read
    // RECOMPUTE: the lane's lines (eta_r, zeta_{2c+h}) inside the cell (padding lanes: weight 0, any point)
    const double eta = c_pts[P][r < n ? r : 0], zeta0 = c_pts[P][v0 ? 2 * c : 0], zeta1 = c_pts[P][v1 ? 2 * c + 1 : 0];
#pragma unroll
    for (int t = 0; t < n; ++t)
    {
      const int o = t * SI + yo[(t >> 1) & 1];
      const double2 g = *reinterpret_cast<const double2*>(B0 + o);
      double w0, w1;
      if constexpr (STREAM || RECOMPUTE)
      {
        double2 qr[6]; // RECOMPUTE: G at the lane's two points of tile t, weights folded in
        if constexpr (RECOMPUTE)
        { // the vertices are re-read from shared memory for every tile (volatile): held in registers across the
          // tiles, the lane's coefficients spill next to gy, gz
          const volatile double* sv = SV;
          double v[8][3];
#pragma unroll
          for (int kk = 0; kk < 8; ++kk)
#pragma unroll
            for (int i = 0; i < 3; ++i)
              v[kk][i] = sv[kk * 3 + i];
          TrilinearMonomials M;
          M.from_vertices(v);
          JacobianAlongXi jac;
          double J[3][3], g0[6], g1[6];
          jac.init(M, eta, zeta0);
          jac.at(c_pts[P][t], J);
          g_from_jacobian(J, literal_detj, c_wts[P][t] * wr0, g0);
          jac.init(M, eta, zeta1);
          jac.at(c_pts[P][t], J);
          g_from_jacobian(J, literal_detj, c_wts[P][t] * wr1, g1);
#pragma unroll
          for (int cc = 0; cc < 6; ++cc)
            qr[cc] = make_double2(g0[cc], g1[cc]);
        }
        else if (t + 1 < n)
          load_g(t + 1, gq[(t + 1) & 1]);
        const double2* q = RECOMPUTE ? qr : gq[t & 1];
        w0 = w1 = kap;
        G00 = q[0].x, G01 = q[1].x, G02 = q[2].x, G11 = q[3].x, G12 = q[4].x, G22 = q[5].x;
        const double f0 = G00 * g.x + G01 * gy[t][0] + G02 * gz[t][0];
        const double f1 = G01 * g.x + G11 * gy[t][0] + G12 * gz[t][0];
        const double f2 = G02 * g.x + G12 * gy[t][0] + G22 * gz[t][0];
        G00 = q[0].y, G01 = q[1].y, G02 = q[2].y, G11 = q[3].y, G12 = q[4].y, G22 = q[5].y;
        *reinterpret_cast<double2*>(B0 + o) = make_double2(w0 * f0, w1 * (G00 * g.y + G01 * gy[t][1] + G02 * gz[t][1]));
        *reinterpret_cast<double2*>(B1 + o) = make_double2(w0 * f1, w1 * (G01 * g.y + G11 * gy[t][1] + G12 * gz[t][1]));
        *reinterpret_cast<double2*>(B2 + o) = make_double2(w0 * f2, w1 * (G02 * g.y + G12 * gy[t][1] + G22 * gz[t][1]));
      }
      else
      {
        w0 = c_wts[P][t] * wr0, w1 = c_wts[P][t] * wr1;
        *reinterpret_cast<double2*>(B0 + o) = make_double2(w0 * (G00 * g.x + G01 * gy[t][0] + G02 * gz[t][0]),
                                                           w1 * (G00 * g.y + G01 * gy[t][1] + G02 * gz[t][1]));
        *reinterpret_cast<double2*>(B1 + o) = make_double2(w0 * (G01 * g.x + G11 * gy[t][0] + G12 * gz[t][0]),
                                                           w1 * (G01 * g.y + G11 * gy[t][1] + G12 * gz[t][1]));
        *reinterpret_cast<double2*>(B2 + o) = make_double2(w0 * (G02 * g.x + G12 * gy[t][0] + G22 * gz[t][0]),
                                                           w1 * (G02 * g.y + G12 * gy[t][1] + G22 * gz[t][1]));
      }
    }
    __syncwarp();
    if constexpr (AHEAD)
      if (pl + nw < count)
        load_idx(pl + nw, dn);
    // ---- transposed contractions
    double ayz[n][2], ax[n][2];
#pragma unroll
    for (int t = 0; t < n; ++t)
    {
      const int b = (t >> 1) & 1;
      ayz[t][0] = ayz[t][1] = ax[t][0] = ax[t][1] = 0.0;
      dmma884(ayz[t][0], ayz[t][1], B2[t * SI + f1[b]], tA0);          // sum_q fz(t,j,q) D[q][k]
      dmma884(ayz[t][0], ayz[t][1], B2[t * SI + (f1[b] ^ 4)], tA1);
      dmma884(ayz[t][0], ayz[t][1], tA0, B1[t * SI + f2[b]]);          // sum_q D[q][j] fy(t,q,k)
      dmma884(ayz[t][0], ayz[t][1], tA1, B1[t * SI + 32 + f2[b]]);
      dmma884(ax[t][0], ax[t][1], tA0, B0[t * 8 + f3[b]]);             // sum_q D[q][i] fx(q,t,k)
      dmma884(ax[t][0], ax[t][1], tA1, B0[t * 8 + 4 * SI + f3[b]]);
    }
    __syncwarp(); // every lane is done reading the fluxes: B1 carries the X accumulator to layout Y
#pragma unroll
    for (int t = 0; t < n; ++t)
      *reinterpret_cast<double2*>(B1 + t * 8 + xo[(t >> 1) & 1]) = make_double2(ax[t][0], ax[t][1]);
    __syncwarp();
#pragma unroll
    for (int t = 0; t < n; ++t)
    {
      const double2 a = *reinterpret_cast<const double2*>(B1 + t * SI + yo[(t >> 1) & 1]);
#pragma unroll
      for (int h = 0; h < 2; ++h)
      {
        const int dd = d[t][h];
        if (dd >= 0)
          atomicAdd(&y[dd], ayz[t][h] + (h ? a.y : a.x));
        else if (n == 8 || (h ? v1 : v0))
          y[~dd] = x[~dd]; // Dirichlet row: y = x (src/laplacian.hpp:273-274); rare, boundary cells only
      }
    }
    // no barrier here: B1 is next written by the flux phase, three barriers into the next cell
    if constexpr (AHEAD)
    {
#pragma unroll
      for (int t = 0; t < n; ++t)
        d[t][0] = dn[t][0], d[t][1] = dn[t][1];
    }
  }
}

// MMA_AFFINE reads Gc (one 6-vector per affine cell), MMA_STREAMED reads G (the COLUMN layout), MMA_RECOMPUTED the mesh
template <int P, int GEO>
struct MmaApply
{
  // WPB warps (cells) per CTA; MINB CTAs per SM the kernel is compiled for.  6 (168 registers, 16 bytes of spills
  // at P7, 12 warps per SM) against 7 (128 registers, 130-180 bytes of spills, 14 warps), measured at 100 M dofs:
  // affine P6 1.42 vs 1.54 ms, P7 1.19 vs 1.38 ms; streamed P6 2.22 vs 2.93 ms, P7 1.76 vs 2.58 ms.  5 compiles to
  // the same code as 6.
  static constexpr int WPB = 2, MINB = 6;
  using C = MmaCfg<P, WPB>;
  static constexpr bool cell_geometry = GEO == MMA_AFFINE;
  static constexpr int cpb = 0;
  static constexpr size_t smem = C::smem + (GEO == MMA_RECOMPUTED ? WPB * 24 * sizeof(double) : 0);
  static void name(char* s, int cap)
  {
    snprintf(s, cap, "k_apply_affine_mma<%d,%d,%s>", P, WPB,
             GEO == MMA_AFFINE ? "affine" : (GEO == MMA_STREAMED ? "streamed" : "recomputed"));
  }
  static void launch(pmgx_ctx* c, cudaStream_t st, const ApplyArgs& a)
  {
    launch_persistent<k_apply_affine_mma<P, WPB, MINB, GEO>>(c, st, a, "k_apply_affine_mma", P, WPB * 32, smem,
                                                              (a.count + WPB - 1) / WPB, a.cell0, a.count, a.xgeom,
                                                              a.geom_dofmap, a.literal_detj);
  }
};
