// CR adaptation: the deterministic reduction helpers of cr_update_kernel (kernels_generic.cuh, which includes this
// header where they used to be defined) and, in the multi-problem NVRTC module only (BPM_JIT_PROBLEMS), the
// per-problem CR kernel built on them.  Device code only.  (The multi-problem kernel lives in that module because a
// second kernel of the library using these helpers would move the static shared arrays of cr_update_kernel.)
#pragma once
#include "step.cuh"

namespace bpm {

// Stage 1: block b sums the chains of its contiguous segment (fixed order inside the
// block); stage 2: one warp adds the block partials in block order.
constexpr int kCrBlocks = 148;
// Second half of the reduction, run by whichever block finishes last (ticket counter): adds
// the block partials in block order -- so the sums do not depend on scheduling -- and, on an
// unsharded handle, applies the p_cr update (dream.py:132-140).  One launch per generation
// instead of three.
__device__ __forceinline__ void cr_apply(const double* __restrict__ part, int n_cr, double* __restrict__ dm,
                                         double* __restrict__ cnt, double* __restrict__ p_cr) {
  double got = 0.0;
  for (int m = 0; m < n_cr; ++m) {
    dm[m] += part[m];
    cnt[m] += part[n_cr + m];
    got += part[n_cr + m];
  }
  if (got == 0.0) return;  // no chain ran _update_cr_ratios this generation
  int nz = 0;
  for (int m = 0; m < n_cr; ++m) nz += cnt[m] > 0.0;
  if (nz == n_cr)
    for (int m = 0; m < n_cr; ++m) p_cr[m] = dm[m] / cnt[m];
  double tot = 0.0;
  for (int m = 0; m < n_cr; ++m) tot += p_cr[m];
  for (int m = 0; m < n_cr; ++m) p_cr[m] /= tot;
}

// first half: block `bid` of `nb` sums the chains of its contiguous segment (256 threads)
__device__ __forceinline__ void cr_block_partials(const double* __restrict__ cr_delta,
                                                  const int32_t* __restrict__ cr_pick, int lo, int hi, int n_cr,
                                                  int bid, int nb, double* __restrict__ block_part) {
  __shared__ double sm[8][2 * 4];
  const int n = hi - lo;
  const int per = (n + nb - 1) / nb;
  const int c0 = lo + bid * per;
  const int c1 = min(hi, c0 + per);
  if (n_cr <= 4) {
    // one pass over the block's chains, the (at most four) CR classes in registers
    double s[4] = {0.0, 0.0, 0.0, 0.0}, k[4] = {0.0, 0.0, 0.0, 0.0};
    // eight independent (pick, statistic) loads in flight per thread, folded in chain order
    for (int base = c0; base < c1; base += 8 * 256) {
      int mm[8];
      double vv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int c = base + u * 256 + (int)threadIdx.x;
        const bool ok = c < c1;
        mm[u] = ok ? cr_pick[c] : -1;
        vv[u] = ok ? cr_delta[c] : 0.0;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (mm[u] == q) { s[q] += vv[u]; k[q] += 1.0; }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        s[q] += __shfl_xor_sync(0xFFFFFFFFu, s[q], o);
        k[q] += __shfl_xor_sync(0xFFFFFFFFu, k[q], o);
      }
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
      for (int q = 0; q < 4; ++q) { sm[threadIdx.x >> 5][q] = s[q]; sm[threadIdx.x >> 5][4 + q] = k[q]; }
    }
    __syncthreads();
    if (threadIdx.x < 8) {
      const int q = threadIdx.x & 3, pass = threadIdx.x >> 2;
      double w = 0.0;
      for (int i = 0; i < 8; ++i) w += sm[i][threadIdx.x];
      if (q < n_cr) block_part[(size_t)bid * 2 * BPM_MAX_CR + pass * n_cr + q] = w;
    }
    __syncthreads();
  } else {
    for (int m = 0; m < n_cr; ++m) {
      double s = 0.0, k = 0.0;
      for (int c = c0 + threadIdx.x; c < c1; c += blockDim.x)
        if (cr_pick[c] == m) { s += cr_delta[c]; k += 1.0; }
      for (int pass = 0; pass < 2; ++pass) {
        double v = pass == 0 ? s : k;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
        if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5][0] = v;
        __syncthreads();
        if (threadIdx.x == 0) {
          double w = 0.0;
          for (int i = 0; i < 8; ++i) w += sm[i][0];
          block_part[(size_t)bid * 2 * BPM_MAX_CR + pass * n_cr + m] = w;
        }
        __syncthreads();
      }
    }
  }
}
// second half, one block: all block partials land in shared memory with independent loads, then each of
// the 2 n_cr outputs is added up in block order
__device__ __forceinline__ void cr_finish(const double* __restrict__ block_part, int nb, int n_cr,
                                          double* __restrict__ part, int apply, double* __restrict__ dm,
                                          double* __restrict__ cnt, double* __restrict__ p_cr) {
  __shared__ double stage[kCrBlocks * 2 * BPM_MAX_CR / 4];    // nb <= 148 blocks x 2 n_cr <= 8 values (n_cr <= 4) or fewer blocks
  const int nv = 2 * n_cr;
  const int fit = (int)(sizeof(stage) / sizeof(double)) / nv;      // blocks that fit in the stage
  double w = 0.0;
  for (int b0 = 0; b0 < nb; b0 += fit) {
    const int nb_here = min(nb - b0, fit);
    for (int idx = threadIdx.x; idx < nb_here * nv; idx += blockDim.x) {
      const int b = idx / nv, i = idx - b * nv;
      stage[idx] = __ldcg(&block_part[(size_t)(b0 + b) * 2 * BPM_MAX_CR + i]);
    }
    __syncthreads();
    if ((int)threadIdx.x < nv)
      for (int b = 0; b < nb_here; ++b) w += stage[b * nv + threadIdx.x];
    __syncthreads();
  }
  __shared__ double part_s[2 * BPM_MAX_CR];        // cr_apply reads the sums from here, not back from global memory
  if ((int)threadIdx.x < nv) {
    part[threadIdx.x] = w;
    part_s[threadIdx.x] = w;
  }
  __syncthreads();
  if (threadIdx.x == 0 && apply) cr_apply(part_s, n_cr, dm, cnt, p_cr);
}

#ifdef BPM_JIT_PROBLEMS
// Grid (nb, P): problem g = blockIdx.y reduces chains [g n, (g + 1) n) with the helpers and the block count
// cr_update_kernel uses on a handle of n chains (nb = min(cdiv(n, 2048), kCrBlocks)), so its sums are added in
// the same order, and applies the p_cr update to its own row [g][BPM_MAX_CR].  One ticket per problem.
__global__ void __launch_bounds__(256) cr_update_problems_kernel(const double* __restrict__ cr_delta,
                                                                 const int32_t* __restrict__ cr_pick, int n, int n_cr,
                                                                 double* __restrict__ block_part,
                                                                 unsigned int* __restrict__ tickets,
                                                                 double* __restrict__ part, double* __restrict__ dm,
                                                                 double* __restrict__ cnt, double* __restrict__ p_cr) {
  __shared__ bool last;
  const int g = blockIdx.y;
  double* bp = block_part + (size_t)g * gridDim.x * 2 * BPM_MAX_CR;
  cr_block_partials(cr_delta, cr_pick, g * n, (g + 1) * n, n_cr, (int)blockIdx.x, (int)gridDim.x, bp);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicAdd(tickets + g, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (threadIdx.x == 0) tickets[g] = 0u;
  const size_t o = (size_t)g * BPM_MAX_CR;
  cr_finish(bp, (int)gridDim.x, n_cr, part + 2 * o, 1, dm + o, cnt + o, p_cr + o);
}
#endif

}  // namespace bpm
