// CSR operator type shared between csr.cu (SpMV) and laplacian.cu (device assembly).
#pragma once
#include "operator.hpp"

namespace pmgx
{
struct CsrOperator : pmgx_operator
{
  long long nnz = 0;
  bool has_ghost_cols = false;
  DevBuf<int32_t> row_ptr;  // n_owned + 1
  DevBuf<int32_t> off_diag; // n_owned: first ghost-column entry of each row (src/csr.hpp:118-121)
  DevBuf<int32_t> cols;
  DevBuf<double> values;
  DevBuf<int32_t> ghost_rows; // rows with at least one ghost-column entry
  int n_ghost_rows = 0;
  void apply(double* x, double* y) override;
  bool supports_cheb_fusion() const override { return true; }
  bool apply_cheb(double* in, const ChebEp& e) override;
  void finish_setup(); // extracts diag^-1 (src/csr.hpp:101-112)
};

// Reduced-storage twin of a CsrOperator for use INSIDE a preconditioner (amg.cu, level 0): the owned-
// column block of the same matrix with FP32 values and, when every owned column lies within +-32767 of
// its row, 16-bit column deltas -- 6 (or 8) bytes per non-zero instead of 12, on a kernel that is purely
// HBM-bound -- stored as SLICED ELL (32-row slices, column-major inside a slice): one thread per row, so
// the value / delta loads of a warp are one contiguous run per step and, on meshes numbered along grid
// lines, so are the gathers of x (consecutive rows hit consecutive columns).  With 8 lanes per CSR row
// the same kernel is bound by the L1 gather rate at half the bytes (measured: 75 us vs 89 us for FP64
// CSR at 40 M non-zeros).  Vectors stay FP64; the (small) ghost-column block stays FP64 CSR.  The
// rounded matrix is still symmetric, so a cycle smoothed with it is a (slightly different) symmetric
// preconditioner; the Krylov operator itself is never replaced.
struct CsrOperatorLP : pmgx_operator
{
  CsrOperator* src = nullptr; // borrowed: ghost rows, FP64 ghost-column block, halo
  bool d16 = false;
  int n_slices = 0;
  DevBuf<long long> slice_ptr; // n_slices + 1: first entry of every slice
  DevBuf<float> vals32;        // [slice_ptr[s] + k * 32 + lane]; padding: value 0, column = the row itself
  DevBuf<int16_t> dcol16;      // col - row (d16) ...
  DevBuf<int32_t> cols32;      // ... or the column itself
  void apply(double* x, double* y) override;
  bool supports_cheb_fusion() const override { return true; }
  bool apply_cheb(double* in, const ChebEp& e) override;
};
CsrOperatorLP* make_lp(CsrOperator* A);
} // namespace pmgx
