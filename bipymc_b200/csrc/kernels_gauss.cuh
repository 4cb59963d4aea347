// Gaussian likelihood with a dense data covariance (BPM_TARGET_JIT_GAUSS): the run-time compiled kernels of the
// kind kJitGauss (engine.cu).  Its translation unit places, before this header, the user's
//   __device__ double model_mean(const double* theta, const double* row);   // E[y_i | theta] at row x_i
//   __device__ double ln_prior(const double* theta);                        // when BPM_HAS_PRIOR is 1
// and defines BPM_DIM, BPM_NROWS (M), BPM_ROWLEN (k) and BPM_HAS_PRIOR.  x is the row-major [M][k] array.
//
// One evaluation of n rows of theta is three launches:
//   1. gauss_model_kernel: Yp[c][i] = model_mean(theta_c, x_i) into a workspace [n][Mp], Mp = M rounded up to a
//      multiple of 16, the padding entries 0.0;
//   2. gauss_data_kernel (gauss_data.cuh, library code): part[cb][c] = the squares of (Yp[c] - y) . B[:, cb],
//      column block cb of 128 columns of B = L^-T (C = L L^T), on the FP64 tensor pipe;
//   3. gauss_lnl_finish_kernel: maha = ((part[0] + part[1]) + part[2]) + ... in cb order, then
//      ln L = ln_prior + (-0.5 (c0 + maha)), -inf when ln_prior is -inf whatever model_mean returned.
// Every addition's order is fixed by M alone, so a given theta gets the same bits whatever the batch.
#pragma once
#include "kernels_sum.cuh"

namespace bpm {

// rows of x per CTA of gauss_model_kernel: one stage of the sum kernels' staging when a row is staged (k <= 8)
__host__ __device__ constexpr int gauss_model_rows(int k) {
  return k <= kSumSmemRowLen ? sum_stage_chunks(k) * kSumChunk : kSumChunk;
}
__host__ __device__ constexpr size_t gauss_model_smem(int k) {
  return k <= kSumSmemRowLen ? sizeof(double) * k * gauss_model_rows(k) : 0;
}
__host__ __device__ constexpr int64_t gauss_rows_padded(int64_t M) { return (M + 15) / 16 * 16; }

#ifdef BPM_JIT_GAUSS
constexpr int64_t kGaussRows = BPM_NROWS;
constexpr int64_t kGaussRowsPad = gauss_rows_padded(kGaussRows);
constexpr int kGaussModelRows = gauss_model_rows(kSumK);

// grid (ceil(n / tile), ceil(Mp / kGaussModelRows)), kSumThreads threads, dynamic shared memory gauss_model_smem(k).
// CTA (t, b) writes rows [t tile, (t + 1) tile) of Yp, columns [b R, (b + 1) R), R = kGaussModelRows, lanes along
// the columns.  n_dev (may be null): rows at or past *n_dev - n_off are skipped.
__global__ void __launch_bounds__(kSumThreads) gauss_model_kernel(const double* __restrict__ P, int n, int ld,
                                                                  const int32_t* __restrict__ n_dev, int n_off,
                                                                  const double* __restrict__ x, int tile,
                                                                  double* __restrict__ Yp) {
  extern __shared__ __align__(16) double sm_gm[];         // [k][kGaussModelRows] when staged
  const int nv = n_dev ? min(n, *n_dev - n_off) : n;
  const int c0 = blockIdx.x * tile;
  if (c0 >= nv) return;
  const int nt = min(tile, nv - c0);
  const int64_t r0 = (int64_t)blockIdx.y * kGaussModelRows;
  if constexpr (kSumStaged) {
    sum_stage(sm_gm, x, r0, min((int64_t)kGaussModelRows, kGaussRows - r0));
    __syncthreads();
  }
  const int nr = (int)min((int64_t)kGaussModelRows, kGaussRowsPad - r0);
  for (int ci = 0; ci < nt; ++ci) {
    SumTheta th;
    th.load(P + (size_t)(c0 + ci) * ld);
    double* __restrict__ yrow = Yp + (size_t)(c0 + ci) * kGaussRowsPad + r0;
    for (int r = threadIdx.x; r < nr; r += kSumThreads) {
      double v = 0.0;
      if (r0 + r < kGaussRows) {
        if constexpr (kSumStaged) {
          double rv[kSumK];
#pragma unroll
          for (int q = 0; q < kSumK; ++q) rv[q] = sm_gm[q * kSumStageRows + r];
          v = model_mean(th.ptr(), rv);
        } else {
          v = model_mean(th.ptr(), x + (r0 + r) * kSumK);
        }
      }
      yrow[r] = v;
    }
  }
}

// Thread per row: part is [n_cb][n] (gauss_data_kernel).  out[c] = ln L.
__global__ void __launch_bounds__(128) gauss_lnl_finish_kernel(const double* __restrict__ P, int n, int ld,
                                                               const int32_t* __restrict__ n_dev, int n_off,
                                                               const double* __restrict__ part, int n_cb, double c0,
                                                               double* __restrict__ out) {
  const int nv = n_dev ? min(n, *n_dev - n_off) : n;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nv) return;
  SumTheta th;
  th.load(P + (size_t)c * ld);
  const double prior = sum_prior(th.ptr());
  double maha = part[c];
  for (int cb = 1; cb < n_cb; ++cb) maha = __dadd_rn(maha, part[(size_t)cb * n + c]);
  out[c] = sum_finish_value(prior, gauss_finish(c0, maha, 0));
}
#endif  // BPM_JIT_GAUSS

}  // namespace bpm
