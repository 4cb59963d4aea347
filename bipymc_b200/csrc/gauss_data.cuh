// Quadratic form of a Gaussian likelihood with a dense data covariance (BPM_TARGET_JIT_GAUSS), on the FP64 tensor
// pipe.  With C = L L^T and B = L^-T (upper triangular, [Mp][Mp] row-major, zero-padded), row c of the model
// predictions Yp [n][Mp] (kernels_gauss.cuh: gauss_model_kernel) has
//   maha_c = | (Yp[c] - y) . B |^2 = sum over column blocks cb of part[cb][c],
// and this kernel writes part [ncb][n], ncb = ceil(Mp / 128).  It is the gauss_dmma_kernel's DMMA tile, ring and
// fold with two changes for few chains and a triangular operand:
//   * the grid is (row tiles, column blocks): CTA (t, cb) computes the 16 MT x 128 tile of column block cb, so
//     n / (16 MT) x ncb CTAs fill the GPU at any chain count.  Row tiles of one column block are adjacent in launch
//     order: they share that block of B while it is in L2;
//   * its k-loop stops at the block's last column, (cb + 1) 128: the rows of B below it are zero, which halves the
//     work.
// y is subtracted on the A-operand load, from a 16-double slice staged with each k tile.  The per-row arithmetic
// (k order of the DMMA accumulators, the fold over a warp's columns, the quad shuffles, the four column warps in
// order) is the same for MT = 2 and 4, so the tile size, chosen from n only, changes no bits.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "gauss_dmma.cuh"

namespace bpm {

__host__ __device__ constexpr size_t gx_stage_doubles(int M) { return gd_stage_doubles(M) + kGdK; }   // + y slice

// n: rows of Yp (and the row stride of part); n_dev (may be null): rows at or past *n_dev - n_off are not computed.
// Mp % 16 == 0.
template <int MT>
__global__ void __launch_bounds__(kGdThreads, 2)
gauss_data_kernel(const double* __restrict__ Yp, int n, int Mp, const int32_t* __restrict__ n_dev, int n_off,
                  const double* __restrict__ y, const double* __restrict__ B, double* __restrict__ part) {
  constexpr int kGdM = 16 * MT;
  int nv = n;
  if (n_dev) {
    nv = min(n, *n_dev - n_off);
    if ((int)blockIdx.x * kGdM >= nv) return;
  }
  constexpr size_t kStage = gx_stage_doubles(kGdM);
  extern __shared__ __align__(16) double gxs[];
  double* ring = gxs;
  double* red = ring + kGdStages * kStage;                     // [4][kGdM] row sums per column-warp
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int wr = warp >> 2, wc = warp & 3;                     // warp tile: rows 8 MT wr, cols 32 wc
  const int lq = lane >> 2, lk = lane & 3;
  const int m0 = blockIdx.x * kGdM;
  const int cb = blockIdx.y;
  const int kend = min(Mp, (cb + 1) * kGdN);                   // rows of B past the block's last column are 0
  const int nkt = kend / kGdK;

  auto issue = [&](int kt) {
    if (kt < nkt) {
      double* As = ring + (size_t)(kt % kGdStages) * kStage;
      double* Bs = As + (size_t)kGdM * kGdLda;
      double* ys = Bs + (size_t)kGdK * kGdLdb;
      for (int c = tid; c < kGdM * (kGdK / 2); c += kGdThreads) {
        const int row = c >> 3, k2 = (c & 7) * 2;
        const int gr = m0 + row;
        const bool ok = gr < nv;
        gd_cp16(As + row * kGdLda + k2, Yp + (size_t)(ok ? gr : 0) * Mp + kt * kGdK + k2, ok);
      }
      for (int c = tid; c < kGdK * (kGdN / 2); c += kGdThreads) {
        const int kk = c >> 6, n2 = (c & 63) * 2;
        const int gn = cb * kGdN + n2;
        const bool ok = gn < Mp;
        gd_cp16(Bs + kk * kGdLdb + n2, B + (size_t)(kt * kGdK + kk) * Mp + (ok ? gn : 0), ok);
      }
      if (tid < kGdK / 2) gd_cp16(ys + 2 * tid, y + kt * kGdK + 2 * tid, true);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  issue(0);
  issue(1);
  double acc[MT][4][2];
#pragma unroll
  for (int i = 0; i < MT; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
  for (int kt = 0; kt < nkt; ++kt) {
    asm volatile("cp.async.wait_group 1;" ::: "memory");       // this step's tiles have landed
    __syncthreads();                                           // ... for every thread; the slot of kt-1 is free
    issue(kt + 2);
    const double* As = ring + (size_t)(kt % kGdStages) * kStage;
    const double* Bs = As + (size_t)kGdM * kGdLda;
    const double* ys = Bs + (size_t)kGdK * kGdLdb;
#pragma unroll
    for (int k4 = 0; k4 < kGdK / 4; ++k4) {
      double af[MT], bf[4];
      const double yk = ys[4 * k4 + lk];
#pragma unroll
      for (int i = 0; i < MT; ++i) af[i] = __dsub_rn(As[(8 * MT * wr + 8 * i + lq) * kGdLda + 4 * k4 + lk], yk);
#pragma unroll
      for (int j = 0; j < 4; ++j) bf[j] = Bs[(4 * k4 + lk) * kGdLdb + 32 * wc + 8 * j + lq];
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) gd_dmma(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  // fold the block's squares: a lane's 8 columns, then the quad lanes, then the 4 column-warps of a row group
#pragma unroll
  for (int i = 0; i < MT; ++i) {
    double v = 0.0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      v = fma(acc[i][j][0], acc[i][j][0], v);
      v = fma(acc[i][j][1], acc[i][j][1], v);
    }
    v += __shfl_xor_sync(0xFFFFFFFFu, v, 1);
    v += __shfl_xor_sync(0xFFFFFFFFu, v, 2);
    if (lk == 0) red[wc * kGdM + 8 * MT * wr + 8 * i + lq] = v;
  }
  __syncthreads();
  if (tid < kGdM) {
    const int row = m0 + tid;
    if (row < nv) {
      double s = red[tid];
      s = __dadd_rn(s, red[kGdM + tid]);
      s = __dadd_rn(s, red[2 * kGdM + tid]);
      s = __dadd_rn(s, red[3 * kGdM + tid]);
      part[(size_t)cb * n + row] = s;
    }
  }
}

inline size_t gauss_data_smem(int M) {
  return sizeof(double) * (kGdStages * gx_stage_doubles(M) + 4 * (size_t)M);
}

template <int MT>
inline int launch_gauss_data_t(const double* Yp, int n, int Mp, const int32_t* n_dev, int n_off, const double* y,
                               const double* B, double* part, cudaStream_t s) {
  constexpr int M = 16 * MT;
  const size_t sm = gauss_data_smem(M);
  if (cudaFuncSetAttribute(gauss_data_kernel<MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) !=
      cudaSuccess)
    return 1;
  gauss_data_kernel<MT><<<dim3((n + M - 1) / M, (Mp + kGdN - 1) / kGdN), kGdThreads, sm, s>>>(Yp, n, Mp, n_dev,
                                                                                             n_off, y, B, part);
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

// The tile size as launch_gauss_dmma chooses it: 64-row tiles once there are enough of them to put two on every
// SM, else 32-row tiles.
inline int launch_gauss_data(const double* Yp, int n, int Mp, const int32_t* n_dev, int n_off, const double* y,
                             const double* B, double* part, cudaStream_t s) {
  const bool small = (n + 63) / 64 < 2 * 148;
  return small ? launch_gauss_data_t<2>(Yp, n, Mp, n_dev, n_off, y, B, part, s)
               : launch_gauss_data_t<4>(Yp, n, Mp, n_dev, n_off, y, B, part, s);
}

}  // namespace bpm
