// Assembled CSR operator for the coarse P1 level (north_star item 5).
// Replaces spmv_impl (src/csr.hpp:20-36) and acc::MatrixOperator::operator()
// (src/csr.hpp:220-273): a sub-warp of 8 lanes per row (P1 hex rows hold <= 27 entries)
// with a shuffle reduction instead of one thread per row; the owned-column block runs while
// the halo is in flight, the ghost-column block after it (same split at off_diag_offset).
#include "common.hpp"
#include "operator.hpp"
#include "csr.hpp"
#include "solvers.hpp"

namespace pmgx
{
namespace
{
constexpr int LPR = 8; // lanes per row
constexpr int ST = 256;

// y[i] (=|+=) sum_{j in [beg[i], end[i])} v[j] x[col[j]]: 8 lanes per row, one row per lane
// group.  Every lane keeps UNR independent (value, column) loads in flight, so the dependent
// chain per row is three loads deep (row bounds -> columns/values -> x) and the matrix stream is
// latency-hidden; values / columns are streamed once (evict-first) so that x and y stay in L2.
// Measured at P1, 1.59 M rows, 40 M non-zeros: 95 us = 5.4 TB/s (scalar loop version: 130 us).
// Fusing the CG inner products into this kernel was tried and dropped: a last-block ticket over
// 49 k CTAs serialises on one atomic (234 us), a grid-stride version with few CTAs is latency-bound.
constexpr int UNR = 4;
template <bool ACCUM>
__global__ void __launch_bounds__(ST)
k_spmv(int n_rows, const double* __restrict__ vals, const int32_t* __restrict__ beg,
       const int32_t* __restrict__ end, const int32_t* __restrict__ cols,
       const double* __restrict__ x, double* __restrict__ y)
{
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int row = gt / LPR, lane = gt % LPR;
  double s = 0.0;
  if (row < n_rows)
  {
    const int e = end[row];
    for (int j0 = beg[row] + lane; j0 < e; j0 += UNR * LPR)
    {
      int c[UNR];
      double v[UNR];
#pragma unroll
      for (int t = 0; t < UNR; ++t)
      {
        const int jj = j0 + t * LPR;
        const bool ok = jj < e;
        c[t] = ok ? __ldcs(cols + jj) : -1;
        v[t] = ok ? __ldcs(vals + jj) : 0.0;
      }
#pragma unroll
      for (int t = 0; t < UNR; ++t)
        if (c[t] >= 0)
          s = fma(v[t], x[c[t]], s);
    }
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1)
    s += __shfl_xor_sync(0xffffffffu, s, o);
  if (row < n_rows && lane == 0)
    y[row] = ACCUM ? y[row] + s : s;
}

// ghost-column block of the rows that have one (the rows of dofs on a partition interface):
// y[row] += sum over [off_diag[row], row_ptr[row+1])
__global__ void __launch_bounds__(ST)
k_spmv_ghost_rows(int n_list, const int32_t* __restrict__ rows, const double* __restrict__ vals,
                  const int32_t* __restrict__ off_diag, const int32_t* __restrict__ row_ptr,
                  const int32_t* __restrict__ cols, const double* __restrict__ x, double* __restrict__ y)
{
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int li = gt / LPR, lane = gt % LPR;
  double s = 0.0;
  int row = -1;
  if (li < n_list)
  {
    row = rows[li];
    const int e = row_ptr[row + 1];
    for (int j = off_diag[row] + lane; j < e; j += LPR)
      s = fma(vals[j], x[cols[j]], s);
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1)
    s += __shfl_xor_sync(0xffffffffu, s, o);
  if (row >= 0 && lane == 0)
    y[row] += s;
}

// ---- Chebyshev update fused into the SpMV (ChebEp, operator.hpp).  Same arithmetic, in the same order,
// as the stand-alone passes k_cheb_init / k_cheb_step / k_cheb_last / k_cheb_step_xonly of solvers.cu.
template <int MODE>
__device__ __forceinline__ void cheb_row(int i, double q, const double* __restrict__ in, const ChebEp& e)
{
  if (MODE == ChebEp::INIT)
  {
    const double rv = q * (-1.0) + e.b[i];
    e.r[i] = rv;
    e.z_out[i] = (rv * e.dinv[i]) * e.c0;
  }
  else if (MODE == ChebEp::LAST)
    e.r[i] = q * (-1.0) + e.r[i];
  else
  {
    const double rv = q * (-1.0) + e.r[i];
    const double zo = in[i];
    const double zs = zo * e.c1;
    const double zv = (rv * e.dinv[i]) * e.c2 + zs;
    if (MODE == ChebEp::STEP)
    {
      e.r[i] = rv;
      e.z_out[i] = zv;
    }
    const double xo = e.defer == 2 ? zo : (e.defer == 1 ? zo * 1.0 + e.x[i] : e.x[i]);
    e.x[i] = zv * 1.0 + xo;
  }
}

// owned-column block; rows that also hold ghost columns park their partial sum in e.scratch and are
// finished by k_spmv_cheb_ghost_rows once the halo is in
template <typename VT, bool D16, int MODE>
__global__ void __launch_bounds__(ST)
k_spmv_cheb(int n_rows, const VT* __restrict__ vals, const int32_t* __restrict__ beg, const int32_t* __restrict__ end,
            const int32_t* __restrict__ row_ptr, const int16_t* __restrict__ dcol, const int32_t* __restrict__ cols,
            const double* __restrict__ x, const ChebEp e)
{
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int row = gt / LPR, lane = gt % LPR;
  double s = 0.0;
  if (row < n_rows)
  {
    const int en = end[row];
    for (int j0 = beg[row] + lane; j0 < en; j0 += UNR * LPR)
    {
      int c[UNR];
      VT v[UNR];
#pragma unroll
      for (int t = 0; t < UNR; ++t)
      {
        const int jj = j0 + t * LPR;
        const bool ok = jj < en;
        c[t] = ok ? (D16 ? row + (int)__ldcs(dcol + jj) : __ldcs(cols + jj)) : -1;
        v[t] = ok ? __ldcs(vals + jj) : VT(0);
      }
#pragma unroll
      for (int t = 0; t < UNR; ++t)
        if (c[t] >= 0)
          s = fma((double)v[t], x[c[t]], s);
    }
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1)
    s += __shfl_xor_sync(0xffffffffu, s, o);
  // the vector update of the CTA's ST / LPR consecutive rows is done by ONE warp with coalesced accesses
  // (lane 0 of every row group doing its own row wastes 7/8 of every sector and every issue slot)
  __shared__ double sq[ST / LPR];
  if (lane == 0)
    sq[threadIdx.x / LPR] = s;
  __syncthreads();
  if (threadIdx.x < ST / LPR)
  {
    const int r = blockIdx.x * (ST / LPR) + threadIdx.x;
    if (r < n_rows)
    {
      if (end[r] < row_ptr[r + 1])
        e.scratch[r] = sq[threadIdx.x]; // ghost columns to come
      else
        cheb_row<MODE>(r, sq[threadIdx.x], x, e);
    }
  }
}

template <int MODE>
__global__ void __launch_bounds__(ST)
k_spmv_cheb_ghost_rows(int n_list, const int32_t* __restrict__ rows, const double* __restrict__ vals,
                       const int32_t* __restrict__ off_diag, const int32_t* __restrict__ row_ptr,
                       const int32_t* __restrict__ cols, const double* __restrict__ x, const ChebEp e)
{
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int li = gt / LPR, lane = gt % LPR;
  double s = 0.0;
  int row = -1;
  if (li < n_list)
  {
    row = rows[li];
    const int en = row_ptr[row + 1];
    for (int j = off_diag[row] + lane; j < en; j += LPR)
      s = fma(vals[j], x[cols[j]], s);
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1)
    s += __shfl_xor_sync(0xffffffffu, s, o);
  if (row >= 0 && lane == 0)
    cheb_row<MODE>(row, e.scratch[row] + s, x, e);
}

template <typename VT, bool D16>
void launch_spmv_cheb(pmgx_ctx* c, int grid, int n_rows, const VT* vals, const int32_t* beg, const int32_t* end,
                      const int32_t* row_ptr, const int16_t* dcol, const int32_t* cols, const double* x, const ChebEp& e)
{
  switch (e.mode)
  {
  case ChebEp::INIT: k_spmv_cheb<VT, D16, ChebEp::INIT><<<grid, ST, 0, c->stream>>>(n_rows, vals, beg, end, row_ptr, dcol, cols, x, e); break;
  case ChebEp::STEP: k_spmv_cheb<VT, D16, ChebEp::STEP><<<grid, ST, 0, c->stream>>>(n_rows, vals, beg, end, row_ptr, dcol, cols, x, e); break;
  case ChebEp::LAST: k_spmv_cheb<VT, D16, ChebEp::LAST><<<grid, ST, 0, c->stream>>>(n_rows, vals, beg, end, row_ptr, dcol, cols, x, e); break;
  default: k_spmv_cheb<VT, D16, ChebEp::XONLY><<<grid, ST, 0, c->stream>>>(n_rows, vals, beg, end, row_ptr, dcol, cols, x, e); break;
  }
  check_launch("k_spmv_cheb");
  count_launch(c);
}

void launch_ghost_rows_cheb(const CsrOperator* A, const double* x, const ChebEp& e)
{
  pmgx_ctx* c = A->ctx;
  const int g2 = (int)(((long long)A->n_ghost_rows * LPR + ST - 1) / ST);
#define PMGX_GR(M)                                                                                                     \
  k_spmv_cheb_ghost_rows<M><<<g2, ST, 0, c->stream>>>(A->n_ghost_rows, A->ghost_rows.p, A->values.p, A->off_diag.p,    \
                                                      A->row_ptr.p, A->cols.p, x, e)
  switch (e.mode)
  {
  case ChebEp::INIT: PMGX_GR(ChebEp::INIT); break;
  case ChebEp::STEP: PMGX_GR(ChebEp::STEP); break;
  case ChebEp::LAST: PMGX_GR(ChebEp::LAST); break;
  default: PMGX_GR(ChebEp::XONLY); break;
  }
#undef PMGX_GR
  check_launch("k_spmv_cheb_ghost_rows");
  count_launch(c);
}

__global__ void k_flag_ghost_rows(int n_rows, const int32_t* __restrict__ off_diag,
                                  const int32_t* __restrict__ row_ptr, int32_t* __restrict__ count,
                                  int32_t* __restrict__ list)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_rows && off_diag[i] < row_ptr[i + 1])
    list[atomicAdd(count, 1)] = i;
}

__global__ void k_extract_diag_inv(int n_rows, const double* __restrict__ vals,
                                   const int32_t* __restrict__ row_ptr,
                                   const int32_t* __restrict__ cols, double* __restrict__ dinv)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_rows)
    return;
  double d = 0.0;
  for (int j = row_ptr[i]; j < row_ptr[i + 1]; ++j)
    if (cols[j] == i)
      d = 1.0 / vals[j]; // src/csr.hpp:104-111
  dinv[i] = d;
}

// ---- reduced-storage sliced-ELL twin (CsrOperatorLP, csr.hpp): thread per row, 32-row slices
constexpr int SLICE = 32;

// sum_k val[slice_ptr[s] + k*32 + lane] * x[col] of the thread's row; the slice width is read once per warp
template <bool D16>
__device__ __forceinline__ double sell_row(int row, int n_rows, const long long* __restrict__ slice_ptr,
                                           const float* __restrict__ vals, const int16_t* __restrict__ dcol,
                                           const int32_t* __restrict__ cols, const double* __restrict__ x)
{
  const int s = row >> 5, lane = row & 31;
  const long long b = slice_ptr[s];
  const int w = (int)((slice_ptr[s + 1] - b) >> 5);
  const float* v = vals + b + lane;
  const int16_t* d = dcol + b + lane;
  const int32_t* c = cols + b + lane;
  const int r = row < n_rows ? row : n_rows - 1; // rows beyond the end only exist as padding of the last slice
  double s0 = 0.0, s1 = 0.0;
  int k = 0;
  for (; k + 4 <= w; k += 4)
  {
    float vv[4];
    int cc[4];
#pragma unroll
    for (int t = 0; t < 4; ++t)
    {
      vv[t] = __ldcs(v + (k + t) * SLICE);
      cc[t] = D16 ? r + (int)__ldcs(d + (k + t) * SLICE) : __ldcs(c + (k + t) * SLICE);
    }
    s0 = fma((double)vv[0], x[cc[0]], s0);
    s1 = fma((double)vv[1], x[cc[1]], s1);
    s0 = fma((double)vv[2], x[cc[2]], s0);
    s1 = fma((double)vv[3], x[cc[3]], s1);
  }
  for (; k < w; ++k)
  {
    const float vv = __ldcs(v + k * SLICE);
    const int cc = D16 ? r + (int)__ldcs(d + k * SLICE) : __ldcs(c + k * SLICE);
    s0 = fma((double)vv, x[cc], s0);
  }
  return s0 + s1;
}

template <bool D16>
__global__ void __launch_bounds__(ST)
k_spmv_sell(int n_rows, const long long* __restrict__ slice_ptr, const float* __restrict__ vals,
            const int16_t* __restrict__ dcol, const int32_t* __restrict__ cols, const double* __restrict__ x,
            double* __restrict__ y)
{
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if ((row >> 5) >= (n_rows + SLICE - 1) / SLICE)
    return;
  const double s = sell_row<D16>(row, n_rows, slice_ptr, vals, dcol, cols, x);
  if (row < n_rows)
    y[row] = s;
}

// the same SpMV with the Chebyshev update as its epilogue: each thread owns a whole row, so no barrier.  Rows that
// also hold ghost columns (off_diag non-null: the operator has some) park their partial sum in e.scratch and are
// finished by k_spmv_cheb_ghost_rows once the halo is in
template <bool D16, int MODE>
__global__ void __launch_bounds__(ST)
k_spmv_sell_cheb(int n_rows, const long long* __restrict__ slice_ptr, const float* __restrict__ vals,
                 const int16_t* __restrict__ dcol, const int32_t* __restrict__ cols,
                 const int32_t* __restrict__ off_diag, const int32_t* __restrict__ row_ptr,
                 const double* __restrict__ x, const ChebEp e)
{
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if ((row >> 5) >= (n_rows + SLICE - 1) / SLICE)
    return;
  const double s = sell_row<D16>(row, n_rows, slice_ptr, vals, dcol, cols, x);
  if (row >= n_rows)
    return;
  if (off_diag && off_diag[row] < row_ptr[row + 1])
    e.scratch[row] = s;
  else
    cheb_row<MODE>(row, s, x, e);
}

// rectangular FP64 sliced-ELL product y (+)= M x (the AMG prolongator: 1..8 entries per row, thread per row)
template <bool ACCUM>
__global__ void __launch_bounds__(ST)
k_spmv_sell_rect(int n_rows, const long long* __restrict__ slice_ptr, const double* __restrict__ vals,
                 const int32_t* __restrict__ cols, const double* __restrict__ x, double* __restrict__ y)
{
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  const int s = row >> 5, lane = row & 31;
  if (row >= n_rows)
    return;
  const long long b = slice_ptr[s];
  const int w = (int)((slice_ptr[s + 1] - b) >> 5);
  const double* v = vals + b + lane;
  const int32_t* c = cols + b + lane;
  double s0 = 0.0, s1 = 0.0;
  int k = 0;
  for (; k + 2 <= w; k += 2)
  {
    const double v0 = __ldcs(v + k * SLICE), v1 = __ldcs(v + (k + 1) * SLICE);
    const int c0 = __ldcs(c + k * SLICE), c1 = __ldcs(c + (k + 1) * SLICE);
    s0 = fma(v0, x[c0], s0);
    s1 = fma(v1, x[c1], s1);
  }
  if (k < w)
    s0 = fma(__ldcs(v + k * SLICE), x[__ldcs(c + k * SLICE)], s0);
  y[row] = ACCUM ? y[row] + (s0 + s1) : s0 + s1;
}

// widths[s] = 32 * max over the slice's rows of the owned-column length; overflow: a delta does not fit 16 bits
__global__ void k_sell_widths(int n_rows, const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ off_diag,
                              const int32_t* __restrict__ cols, long long* __restrict__ widths, int* __restrict__ overflow)
{
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  int len = 0;
  bool ovf = false;
  if (row < n_rows)
  {
    len = off_diag[row] - row_ptr[row];
    for (int j = row_ptr[row]; j < off_diag[row]; ++j)
    {
      const int dlt = cols[j] - row;
      ovf = ovf || dlt > 32767 || dlt < -32767;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
    len = max(len, __shfl_xor_sync(0xffffffffu, len, o));
  if (__any_sync(0xffffffffu, ovf) && (threadIdx.x & 31) == 0)
    atomicOr(overflow, 1);
  if ((threadIdx.x & 31) == 0 && row < n_rows)
    widths[row >> 5] = (long long)len * SLICE;
}

__global__ void k_sell_fill(int n_rows, const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ off_diag,
                            const int32_t* __restrict__ cols, const double* __restrict__ vals,
                            const long long* __restrict__ slice_ptr, float* __restrict__ v32, int16_t* __restrict__ d16,
                            int32_t* __restrict__ c32)
{
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  const int s = row >> 5, lane = row & 31;
  if (s >= (n_rows + SLICE - 1) / SLICE)
    return;
  const long long b = slice_ptr[s];
  const int w = (int)((slice_ptr[s + 1] - b) >> 5);
  const int r = row < n_rows ? row : n_rows - 1;
  const int beg = row < n_rows ? row_ptr[row] : 0, len = row < n_rows ? off_diag[row] - row_ptr[row] : 0;
  for (int k = 0; k < w; ++k)
  {
    const long long p = b + (long long)k * SLICE + lane;
    const bool ok = k < len;
    v32[p] = ok ? (float)vals[beg + k] : 0.f;
    const int col = ok ? cols[beg + k] : r;
    if (d16)
      d16[p] = (int16_t)(col - r);
    if (c32)
      c32[p] = col;
  }
}

// rectangular product for the AMG transfer operators: same kernel body with LANES lanes per row
template <int LANES, bool ACCUM>
__global__ void __launch_bounds__(ST)
k_spmv_rect(int n_rows, const double* __restrict__ vals, const int32_t* __restrict__ ptr,
            const int32_t* __restrict__ cols, const double* __restrict__ x, double* __restrict__ y)
{
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int row = gt / LANES, lane = gt % LANES;
  double s = 0.0;
  if (row < n_rows)
  {
    const int e = ptr[row + 1];
    for (int j = ptr[row] + lane; j < e; j += LANES)
      s = fma(vals[j], x[cols[j]], s);
  }
#pragma unroll
  for (int o = LANES / 2; o > 0; o >>= 1)
    s += __shfl_xor_sync(0xffffffffu, s, o);
  if (row < n_rows && lane == 0)
    y[row] = ACCUM ? y[row] + s : s;
}
} // namespace

void spmv_sell_rect(pmgx_ctx* c, int n_rows, const long long* slice_ptr, const int32_t* cols, const double* vals,
                    const double* x, double* y, bool accumulate)
{
  if (n_rows <= 0)
    return;
  const int grid = (n_rows + ST - 1) / ST;
  if (accumulate)
    k_spmv_sell_rect<true><<<grid, ST, 0, c->stream>>>(n_rows, slice_ptr, vals, cols, x, y);
  else
    k_spmv_sell_rect<false><<<grid, ST, 0, c->stream>>>(n_rows, slice_ptr, vals, cols, x, y);
  check_launch("k_spmv_sell_rect");
  count_launch(c);
}

void spmv_rect(pmgx_ctx* c, int n_rows, const int32_t* row_ptr, const int32_t* cols, const double* vals,
               const double* x, double* y, bool accumulate, int lanes)
{
  if (n_rows <= 0)
    return;
  const int grid = (int)(((long long)n_rows * lanes + ST - 1) / ST);
  if (lanes == 32)
  {
    if (accumulate)
      k_spmv_rect<32, true><<<grid, ST, 0, c->stream>>>(n_rows, vals, row_ptr, cols, x, y);
    else
      k_spmv_rect<32, false><<<grid, ST, 0, c->stream>>>(n_rows, vals, row_ptr, cols, x, y);
  }
  else if (lanes == 4)
  {
    if (accumulate)
      k_spmv_rect<4, true><<<grid, ST, 0, c->stream>>>(n_rows, vals, row_ptr, cols, x, y);
    else
      k_spmv_rect<4, false><<<grid, ST, 0, c->stream>>>(n_rows, vals, row_ptr, cols, x, y);
  }
  else
  {
    if (accumulate)
      k_spmv_rect<8, true><<<grid, ST, 0, c->stream>>>(n_rows, vals, row_ptr, cols, x, y);
    else
      k_spmv_rect<8, false><<<grid, ST, 0, c->stream>>>(n_rows, vals, row_ptr, cols, x, y);
  }
  check_launch("k_spmv_rect");
  count_launch(c);
}

void CsrOperator::apply(double* x, double* y)
{
  cudaSetDevice(ctx->device);
  const int grid = (int)(((long long)n_owned * LPR + ST - 1) / ST);
  // ghost entries of y are zeroed like y.set(0) (src/csr.hpp:225)
  if (n_ghost > 0)
    vec::set(ctx, y + n_owned, n_ghost, 0.0);
  if (halo)
    halo_fwd_begin(halo, x);                                                       // :255
  if (n_owned > 0)
  {
    k_spmv<false><<<grid, ST, 0, ctx->stream>>>(n_owned, values.p, row_ptr.p, off_diag.p, cols.p, x, y); // :256-260
    check_launch("k_spmv");
    count_launch(ctx);
  }
  if (halo)
    halo_fwd_end(halo, x);                                                         // :262
  if (n_ghost_rows > 0)
  {
    // :264-268, restricted to the rows that own a ghost-column entry
    const int g2 = (int)(((long long)n_ghost_rows * LPR + ST - 1) / ST);
    k_spmv_ghost_rows<<<g2, ST, 0, ctx->stream>>>(n_ghost_rows, ghost_rows.p, values.p, off_diag.p, row_ptr.p, cols.p,
                                                  x, y);
    check_launch("k_spmv_ghost_rows");
    count_launch(ctx);
  }
}

// fused apply + Chebyshev update: owned-column block (overlapping the halo) finishes the rows without
// ghost columns, the interface rows are finished behind the exchange
bool CsrOperator::apply_cheb(double* in, const ChebEp& e)
{
  cudaSetDevice(ctx->device);
  PMGX_REQUIRE(n_ghost_rows == 0 || e.scratch, "apply_cheb: scratch vector missing");
  const int grid = (int)(((long long)n_owned * LPR + ST - 1) / ST);
  if (halo)
    halo_fwd_begin(halo, in);
  if (n_owned > 0)
    launch_spmv_cheb<double, false>(ctx, grid, n_owned, values.p, row_ptr.p, off_diag.p, row_ptr.p, nullptr, cols.p, in, e);
  if (halo)
    halo_fwd_end(halo, in);
  if (n_ghost_rows > 0)
    launch_ghost_rows_cheb(this, in, e);
  return true;
}

namespace
{
template <bool D16>
void launch_sell_cheb(const CsrOperatorLP* L, const double* x, const ChebEp& e)
{
  const CsrOperator* A = L->src;
  const int grid = (L->n_slices * SLICE + ST - 1) / ST;
  const int32_t* od = A->n_ghost_rows > 0 ? A->off_diag.p : nullptr;
#define PMGX_SC(M)                                                                                                     \
  k_spmv_sell_cheb<D16, M><<<grid, ST, 0, L->ctx->stream>>>(L->n_owned, L->slice_ptr.p, L->vals32.p, L->dcol16.p,       \
                                                            L->cols32.p, od, A->row_ptr.p, x, e)
  switch (e.mode)
  {
  case ChebEp::INIT: PMGX_SC(ChebEp::INIT); break;
  case ChebEp::STEP: PMGX_SC(ChebEp::STEP); break;
  case ChebEp::LAST: PMGX_SC(ChebEp::LAST); break;
  default: PMGX_SC(ChebEp::XONLY); break;
  }
#undef PMGX_SC
  check_launch("k_spmv_sell_cheb");
  count_launch(L->ctx);
}
} // namespace

void CsrOperatorLP::apply(double* x, double* y)
{
  cudaSetDevice(ctx->device);
  if (n_ghost > 0)
    vec::set(ctx, y + n_owned, n_ghost, 0.0);
  if (halo)
    halo_fwd_begin(halo, x);
  if (n_owned > 0)
  {
    const int grid = (n_slices * SLICE + ST - 1) / ST;
    if (d16)
      k_spmv_sell<true><<<grid, ST, 0, ctx->stream>>>(n_owned, slice_ptr.p, vals32.p, dcol16.p, nullptr, x, y);
    else
      k_spmv_sell<false><<<grid, ST, 0, ctx->stream>>>(n_owned, slice_ptr.p, vals32.p, nullptr, cols32.p, x, y);
    check_launch("k_spmv_sell");
    count_launch(ctx);
  }
  if (halo)
    halo_fwd_end(halo, x);
  if (src->n_ghost_rows > 0)
  {
    // the (small) ghost-column block stays FP64 CSR
    const int g2 = (int)(((long long)src->n_ghost_rows * LPR + ST - 1) / ST);
    k_spmv_ghost_rows<<<g2, ST, 0, ctx->stream>>>(src->n_ghost_rows, src->ghost_rows.p, src->values.p, src->off_diag.p,
                                                  src->row_ptr.p, src->cols.p, x, y);
    check_launch("k_spmv_ghost_rows");
    count_launch(ctx);
  }
}

// fused apply + Chebyshev update, split like CsrOperator::apply_cheb: the owned block (overlapping the halo)
// finishes the rows without ghost columns, the FP64 ghost block of src finishes the others behind the exchange
bool CsrOperatorLP::apply_cheb(double* in, const ChebEp& e)
{
  cudaSetDevice(ctx->device);
  PMGX_REQUIRE(src->n_ghost_rows == 0 || e.scratch, "apply_cheb: scratch vector missing");
  if (halo)
    halo_fwd_begin(halo, in);
  if (n_owned > 0)
  {
    if (d16)
      launch_sell_cheb<true>(this, in, e);
    else
      launch_sell_cheb<false>(this, in, e);
  }
  if (halo)
    halo_fwd_end(halo, in);
  if (src->n_ghost_rows > 0)
    launch_ghost_rows_cheb(src, in, e);
  return true;
}

CsrOperatorLP* make_lp(CsrOperator* A)
{
  pmgx_ctx* c = A->ctx;
  std::unique_ptr<CsrOperatorLP> L(new CsrOperatorLP());
  L->ctx = c;
  L->kind = pmgx_operator::CSR;
  L->n_owned = A->n_owned;
  L->n_ghost = A->n_ghost;
  L->halo = A->halo;
  L->src = A;
  L->diag_inv.alloc((size_t)A->n_owned);
  if (A->n_owned > 0)
    PMGX_CUDA(cudaMemcpyAsync(L->diag_inv.p, A->diag_inv.p, (size_t)A->n_owned * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  const int n = A->n_owned;
  L->n_slices = (n + SLICE - 1) / SLICE;
  L->slice_ptr.alloc((size_t)L->n_slices + 1);
  PMGX_CUDA(cudaMemsetAsync(L->slice_ptr.p, 0, ((size_t)L->n_slices + 1) * sizeof(long long), c->stream));
  DevBuf<int> ovf;
  ovf.alloc(1);
  PMGX_CUDA(cudaMemsetAsync(ovf.p, 0, sizeof(int), c->stream));
  long long total = 0;
  if (n > 0)
  {
    // widths into slice_ptr[1..], then an inclusive prefix sum on the host (n_slices is ~50 k: set-up)
    k_sell_widths<<<(n + ST - 1) / ST, ST, 0, c->stream>>>(n, A->row_ptr.p, A->off_diag.p, A->cols.p, L->slice_ptr.p + 1, ovf.p);
    check_launch("k_sell_widths");
    std::vector<long long> sp((size_t)L->n_slices + 1, 0);
    PMGX_CUDA(cudaMemcpyAsync(sp.data(), L->slice_ptr.p, sp.size() * sizeof(long long), cudaMemcpyDeviceToHost, c->stream));
    PMGX_CUDA(cudaStreamSynchronize(c->stream));
    for (size_t i = 1; i < sp.size(); ++i)
      sp[i] += sp[i - 1];
    total = sp.back();
    PMGX_CUDA(cudaMemcpyAsync(L->slice_ptr.p, sp.data(), sp.size() * sizeof(long long), cudaMemcpyHostToDevice, c->stream));
    PMGX_CUDA(cudaStreamSynchronize(c->stream));
  }
  int o = 0;
  PMGX_CUDA(cudaMemcpyAsync(&o, ovf.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  PMGX_CUDA(cudaStreamSynchronize(c->stream));
  L->d16 = o == 0;
  const size_t cap = (size_t)std::max<long long>(total, 1);
  L->vals32.alloc(cap);
  if (L->d16)
    L->dcol16.alloc(cap);
  else
    L->cols32.alloc(cap);
  if (n > 0)
  {
    k_sell_fill<<<(L->n_slices * SLICE + ST - 1) / ST, ST, 0, c->stream>>>(n, A->row_ptr.p, A->off_diag.p, A->cols.p, A->values.p,
                                                                         L->slice_ptr.p, L->vals32.p, L->dcol16.p, L->cols32.p);
    check_launch("k_sell_fill");
    PMGX_CUDA(cudaStreamSynchronize(c->stream));
  }
  return L.release();
}

void CsrOperator::finish_setup()
{
  n_ghost_rows = 0;
  if (n_owned > 0 && has_ghost_cols)
  {
    DevBuf<int32_t> count;
    count.alloc(1);
    ghost_rows.alloc((size_t)n_owned);
    PMGX_CUDA(cudaMemsetAsync(count.p, 0, sizeof(int32_t), ctx->stream));
    k_flag_ghost_rows<<<(n_owned + 255) / 256, 256, 0, ctx->stream>>>(n_owned, off_diag.p, row_ptr.p, count.p,
                                                                      ghost_rows.p);
    check_launch("k_flag_ghost_rows");
    PMGX_CUDA(cudaMemcpyAsync(&n_ghost_rows, count.p, sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PMGX_CUDA(cudaStreamSynchronize(ctx->stream));
    // the compaction order is arbitrary; every row appears once, so the result does not depend on it
  }
  diag_inv.alloc((size_t)n_owned);
  if (n_owned > 0)
  {
    k_extract_diag_inv<<<(n_owned + 255) / 256, 256, 0, ctx->stream>>>(n_owned, values.p, row_ptr.p,
                                                                       cols.p, diag_inv.p);
    check_launch("k_extract_diag_inv");
    count_launch(ctx);
    PMGX_CUDA(cudaStreamSynchronize(ctx->stream));
  }
}
} // namespace pmgx

using pmgx::CsrOperator;

extern "C"
{
int pmgx_csr_create(pmgx_ctx* ctx, int n_rows, int n_ghost, const int32_t* row_ptr_h,
                    const int32_t* off_diag_offset_h, const int32_t* cols_h, const double* values_h,
                    pmgx_halo* halo, pmgx_operator** out)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(ctx && out && row_ptr_h, "csr_create: null argument");
  PMGX_REQUIRE(n_rows >= 0 && n_ghost >= 0, "csr_create: bad sizes");
  PMGX_CUDA(cudaSetDevice(ctx->device));
  const long long nnz = row_ptr_h[n_rows];
  PMGX_REQUIRE(row_ptr_h[0] == 0 && nnz >= 0, "csr_create: bad row_ptr");
  bool ghost_cols = false;
  for (int i = 0; i < n_rows; ++i)
  {
    PMGX_REQUIRE(row_ptr_h[i] <= off_diag_offset_h[i] && off_diag_offset_h[i] <= row_ptr_h[i + 1],
                 "csr_create: off_diag_offset outside its row");
    ghost_cols = ghost_cols || off_diag_offset_h[i] < row_ptr_h[i + 1];
  }
  for (long long j = 0; j < nnz; ++j)
    PMGX_REQUIRE(cols_h[j] >= 0 && cols_h[j] < n_rows + n_ghost, "csr_create: column out of range");
  std::unique_ptr<CsrOperator> A(new CsrOperator());
  A->ctx = ctx;
  A->kind = pmgx_operator::CSR;
  A->n_owned = n_rows;
  A->n_ghost = n_ghost;
  A->halo = halo;
  A->nnz = nnz;
  A->has_ghost_cols = ghost_cols;
  A->row_ptr.upload(row_ptr_h, (size_t)n_rows + 1, ctx->stream);
  A->off_diag.upload(off_diag_offset_h, (size_t)n_rows, ctx->stream);
  A->cols.upload(cols_h, (size_t)nnz, ctx->stream);
  A->values.upload(values_h, (size_t)nnz, ctx->stream);
  A->finish_setup();
  *out = A.release();
  PMGX_API_END
}

long long pmgx_csr_nnz(pmgx_operator* op)
{
  if (!op || op->kind != pmgx_operator::CSR)
    return -1;
  return static_cast<CsrOperator*>(op)->nnz;
}

int pmgx_csr_get(pmgx_operator* op, int32_t* row_ptr_h, int32_t* cols_h, double* values_h)
{
  PMGX_API_BEGIN
  PMGX_REQUIRE(op && op->kind == pmgx_operator::CSR, "csr_get: not a CSR operator");
  auto* A = static_cast<CsrOperator*>(op);
  PMGX_CUDA(cudaSetDevice(A->ctx->device));
  PMGX_CUDA(cudaStreamSynchronize(A->ctx->stream));
  if (row_ptr_h)
    PMGX_CUDA(cudaMemcpy(row_ptr_h, A->row_ptr.p, ((size_t)A->n_owned + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost));
  if (cols_h && A->nnz > 0)
    PMGX_CUDA(cudaMemcpy(cols_h, A->cols.p, (size_t)A->nnz * sizeof(int32_t), cudaMemcpyDeviceToHost));
  if (values_h && A->nnz > 0)
    PMGX_CUDA(cudaMemcpy(values_h, A->values.p, (size_t)A->nnz * sizeof(double), cudaMemcpyDeviceToHost));
  PMGX_API_END
}
}
