// Per-observation likelihoods summed across the whole GPU (BPM_TARGET_JIT_SUM).  Device code only: the
// run-time compiled translation units of a sum-form source (engine.cu: kJitSum, kJitSumProblems, kJitSumRagged)
// are the only ones that compile its kernels.  Each places, before this header, the user's
//   __device__ double ln_like_term(const double* theta, const double* row);   // one observation
//   __device__ double ln_prior(const double* theta);                          // when BPM_HAS_PRIOR is 1
// and defines BPM_DIM, BPM_NROWS (M), BPM_ROWLEN (k) and BPM_HAS_PRIOR.  data is the row-major [M][k] array.
// The ragged kind (BPM_JIT_SUM_RAGGED instead of BPM_JIT_SUM) has no BPM_NROWS: its problems' M differ and are
// read at run time.
//
// Summation order -- a function of M alone (never of the number of chains, the batch, the launch shape or the
// number of GPUs), so a given theta always gets the same bits:
//   1. rows are cut into chunks of kSumChunk = 256 consecutive rows; the last chunk is padded with terms 0.0;
//   2. inside a chunk, a halving pairwise tree: a[i] += a[i + w/2] for i < w/2, w = 256, 128, ..., 2;
//   3. the chunk partials, padded with 0.0 to the next power of two P2 >= ceil(M / 256), are added by an
//      adjacent-pair tree: p[i] = p[2i] + p[2i+1], level by level, down to one value S;
//   4. ln L = ln_prior(theta) + S when BPM_HAS_PRIOR (-inf when ln_prior is -inf: no term is evaluated), else S.
// In numpy (tests/test_cuda_sum_likelihood_cpu.py: sum_order):
//   a = zeros((nc, 256)); a.flat[:M] = terms;  while a.shape[1] > 1: a = a[:, :w/2] + a[:, w/2:]
//   p = zeros(P2); p[:nc] = a[:, 0];            while p.size > 1:     p = p[0::2] + p[1::2]
//
// Work split: a CTA of 8 warps owns (a tile of up to 64 chains, a group of G consecutive chunks), G a power of
// two, so its chunks are one aligned subtree of step 3.  Rows are staged in shared memory, column-major,
// kSumStageChunks chunks at a time; warp w takes the tile's chains w, w + 8, ... and, for each, every staged
// chunk: lane l evaluates rows l + 32 j (j = 0..7) with a register copy of the row and adds them in the order of
// step 2 (in-lane j / j + 4, j / j + 2, j / j + 1, then an xor butterfly over lanes 16, 8, 4, 2, 1).  Chunk
// partials merge into a per-chain binary-counter stack in shared memory that yields the group's subtree value.
// With one group the CTA writes ln L; otherwise group partials go to a workspace [n_groups][n] and
// lnl_sum_finish_kernel completes step 3 over them.  Chunks and groups past the last one holding rows are
// never evaluated: sum_flush makes the adds their 0.0 leaves would have made.  Only the
// tile size and G depend on the number of rows (engine.cu: sum_plan); the arithmetic does not.
#pragma once
#include "targets.cuh"

namespace bpm {

constexpr int kSumChunk = 256;                 // rows per chunk: 8 per lane of a warp
constexpr int kSumThreads = 256;               // 8 warps
constexpr int kSumMaxTile = 64;                // chains per CTA
constexpr int kSumMaxDepth = 24;               // binary-counter stack depth: G <= 2^23 chunks
constexpr int kSumSmemRowLen = 8;              // rows of up to this many doubles are staged in shared memory

// chunks staged per __syncthreads (4 KB .. 16 KB of rows), and the dynamic shared memory of lnl_sum_kernel:
// per chain a stack of kSumMaxDepth partials and its prior, then the staged rows
__host__ __device__ constexpr int sum_stage_chunks(int k) { return k <= 2 ? 4 : (k <= 4 ? 2 : 1); }
__host__ __device__ constexpr size_t sum_smem_bytes(int tile, int k) {
  return sizeof(double) * ((size_t)tile * (kSumMaxDepth + 1) +
                           (k <= kSumSmemRowLen ? (size_t)k * sum_stage_chunks(k) * kSumChunk : 0));
}

// The Gaussian kind (BPM_JIT_GAUSS, kernels_gauss.cuh) shares the row staging, SumTheta and the prior helpers.
#if defined(BPM_JIT_SUM) || defined(BPM_JIT_SUM_RAGGED) || defined(BPM_JIT_GAUSS)
constexpr int kSumK = BPM_ROWLEN;
constexpr bool kSumStaged = kSumK <= kSumSmemRowLen;
constexpr int kSumStageChunks = sum_stage_chunks(kSumK);
constexpr int kSumStageRows = kSumStageChunks * kSumChunk;

// theta in registers for small d (the compiler hoists the theta-only parts of ln_like_term out of the row loop)
struct SumTheta {
#if BPM_DIM <= 32
  double v[BPM_DIM];
  __device__ __forceinline__ void load(const double* __restrict__ p) {
#pragma unroll
    for (int q = 0; q < BPM_DIM; ++q) v[q] = p[q];
  }
  __device__ __forceinline__ const double* ptr() const { return v; }
#else
  const double* v;
  __device__ __forceinline__ void load(const double* __restrict__ p) { v = p; }
  __device__ __forceinline__ const double* ptr() const { return v; }
#endif
};

__device__ __forceinline__ double sum_prior(const double* theta) {
#if BPM_HAS_PRIOR
  return ln_prior(theta);
#else
  (void)theta;
  return 0.0;
#endif
}

// ln L from the prior and the sum S (step 4)
__device__ __forceinline__ double sum_finish_value(double prior, double S) {
#if BPM_HAS_PRIOR
  return prior == -INFINITY ? -INFINITY : prior + S;
#else
  (void)prior;
  return S;
#endif
}

// Stage rows [r0, r0 + nr) of data[][k] into srows, column-major [k][kSumStageRows], by a CTA of kSumThreads threads
__device__ __forceinline__ void sum_stage(double* srows, const double* __restrict__ data, int64_t r0, int64_t nr) {
  for (int64_t i = threadIdx.x; i < nr * kSumK; i += kSumThreads) {
    const int64_t r = i / kSumK;
    srows[(i - r * kSumK) * kSumStageRows + r] = data[r0 * kSumK + i];
  }
}
#endif  // BPM_JIT_SUM || BPM_JIT_SUM_RAGGED || BPM_JIT_GAUSS

#if defined(BPM_JIT_SUM) || defined(BPM_JIT_SUM_RAGGED)
// Chunk `chunk` (global index) of one chain of data[n_rows][k]: steps 1-2; every lane returns the same value.
// srows: the stage's rows, column-major [k][kSumStageRows], starting at row r0 (staged) -- or nullptr: rows from
// global memory.
__device__ __forceinline__ double sum_chunk(const double* theta, int64_t chunk, const double* srows, int64_t r0,
                                            const double* __restrict__ data, int64_t n_rows, int lane) {
  auto term = [&](int64_t row) -> double {
    if constexpr (kSumStaged) {
      double rv[kSumK];
      const int r = (int)(row - r0);
#pragma unroll
      for (int q = 0; q < kSumK; ++q) rv[q] = srows[q * kSumStageRows + r];
      return ln_like_term(theta, rv);
    } else {
      return ln_like_term(theta, data + row * kSumK);
    }
  };
  const int64_t base = chunk * kSumChunk + lane;
  double t[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) t[j] = base + 32 * j < n_rows ? term(base + 32 * j) : 0.0;
#pragma unroll
  for (int j = 0; j < 4; ++j) t[j] = t[j] + t[j + 4];
#pragma unroll
  for (int j = 0; j < 2; ++j) t[j] = t[j] + t[j + 2];
  double p = t[0] + t[1];
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) p = p + __shfl_xor_sync(0xFFFFFFFFu, p, o);
  return p;
}

// Push the partial of leaf i (0-based inside an aligned subtree) onto a binary-counter stack: the adjacent-pair
// tree of step 3.  After leaves 0 .. 2^g - 1 the subtree's value is stk[g].
__device__ __forceinline__ double sum_merge(const double* stk, int64_t i, double p, int* lvl) {
  int l = 0;
  while ((i >> l) & 1) {
    p = stk[l] + p;
    ++l;
  }
  *lvl = l;
  return p;
}

// Value of a subtree of 2^g leaves of which only the first m (>= 1) were pushed, the rest being 0.0: the adds the
// pushes of the zero leaves would make, without making them (an all-zero subtree is +0.0).
__device__ __forceinline__ double sum_flush(const double* stk, int64_t m, int g) {
  if (m == ((int64_t)1 << g)) return stk[g];
  double p = 0.0;
  for (int l = 0; l < g; ++l) p = ((m >> l) & 1) ? stk[l] + p : p + 0.0;
  return p;
}

__device__ __forceinline__ void sum_push(double* stk, int64_t i, double p, int lane) {
  int lvl;
  p = sum_merge(stk, i, p, &lvl);
  __syncwarp();
  if (lane == 0) stk[lvl] = p;
  __syncwarp();
}
// Step 3 above the groups, by the whole warp of row c: the n_groups partials ws[i n + c] are the first leaves of a
// tree of 2^log2_groups (= P2 / G) leaves, the rest 0.0.  Lane l reduces the aligned block of leaves
// [l B, (l + 1) B), B = max(1, 2^log2_groups / 32), by the binary-counter stack; an adjacent-pair shuffle tree
// (lane l + off into lane l) adds the blocks.  Lane 0 returns the tree's value.
__device__ __forceinline__ double sum_groups(const double* __restrict__ ws, int n, int c, int n_groups,
                                             int log2_groups, int lane) {
  const int lb = log2_groups > 5 ? log2_groups - 5 : 0;     // log2 of the leaves per lane
  const int64_t B = (int64_t)1 << lb;
  const int64_t first = (int64_t)lane * B;
  const int64_t m = max((int64_t)0, min(B, (int64_t)n_groups - first));
  double v = 0.0;                                            // an all-zero block is +0.0
  if (m > 0) {
    double stk[kSumMaxDepth];
    for (int64_t i = 0; i < m; ++i) {
      int lvl;
      const double p = sum_merge(stk, i, ws[(size_t)(first + i) * n + c], &lvl);
      stk[lvl] = p;
    }
    v = sum_flush(stk, m, lb);
  }
  for (int off = 1; off < (1 << (log2_groups - lb)); off <<= 1) {
    const double o = __shfl_down_sync(0xFFFFFFFFu, v, off);
    if ((lane & (2 * off - 1)) == 0) v = v + o;
  }
  return v;
}
#endif  // BPM_JIT_SUM || BPM_JIT_SUM_RAGGED

#ifdef BPM_JIT_SUM
constexpr int64_t kSumRows = BPM_NROWS;
constexpr int64_t kSumChunks = (kSumRows + kSumChunk - 1) / kSumChunk;

// grid (ceil(n / tile), n_groups), kSumThreads threads; dynamic shared memory sum_smem_bytes(tile) (engine.cu).
// P: rows [n][ld]; n_dev (may be null): device-side count of valid rows, rows past it are skipped.
// n_groups == 1: out[c] = ln L; else ws[g * n + c] = the partial of group g.
__global__ void __launch_bounds__(kSumThreads) lnl_sum_kernel(const double* __restrict__ P, int n, int ld,
                                                              const int32_t* __restrict__ n_dev,
                                                              const double* __restrict__ data, int tile,
                                                              int log2_group, int n_groups, double* __restrict__ ws,
                                                              double* __restrict__ out) {
  extern __shared__ __align__(16) double sm_sum[];
  const int nv = n_dev ? min(n, *n_dev) : n;
  const int c0 = blockIdx.x * tile;
  if (c0 >= nv) return;
  const int nt = min(tile, nv - c0);
  double* stk = sm_sum;                                  // [tile][kSumMaxDepth]
  double* prior = stk + tile * kSumMaxDepth;             // [tile]
  double* srows = prior + tile;                          // [k][kSumStageRows] when staged
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t G = (int64_t)1 << log2_group;
  const int64_t q0 = (int64_t)blockIdx.y * G;            // first chunk of the group
  for (int ci = threadIdx.x; ci < nt; ci += kSumThreads) {
    SumTheta th;
    th.load(P + (size_t)(c0 + ci) * ld);
    prior[ci] = sum_prior(th.ptr());
  }
  __syncthreads();
  const int64_t m = min(G, kSumChunks - q0);            // chunks of the group that hold rows (>= 1)
  const int sc = G < kSumStageChunks ? (int)G : kSumStageChunks;
  for (int64_t s0 = 0; s0 < m; s0 += sc) {
    const int64_t r0 = (q0 + s0) * kSumChunk;            // first row of the stage
    const int ns = (int)min((int64_t)sc, m - s0);
    if constexpr (kSumStaged) {
      __syncthreads();                                   // the previous stage's rows are no longer read
      sum_stage(srows, data, r0, min((int64_t)ns * kSumChunk, kSumRows - r0));
      __syncthreads();
    }
    for (int ci = warp; ci < nt; ci += kSumThreads / 32) {
      if (prior[ci] == -INFINITY) continue;              // outside the prior: no term is evaluated
      double* cs = stk + ci * kSumMaxDepth;
      SumTheta th;
      th.load(P + (size_t)(c0 + ci) * ld);
      for (int s = 0; s < ns; ++s)
        sum_push(cs, s0 + s, sum_chunk(th.ptr(), q0 + s0 + s, srows, r0, data, kSumRows, lane), lane);
    }
  }
  __syncthreads();
  for (int ci = threadIdx.x; ci < nt; ci += kSumThreads) {
    const double S = sum_flush(stk + ci * kSumMaxDepth, m, log2_group);
    if (n_groups == 1) out[c0 + ci] = sum_finish_value(prior[ci], S);
    else ws[(size_t)blockIdx.y * n + c0 + ci] = S;
  }
}

// Step 3 above the groups and step 4, one warp per row (sum_groups).
__global__ void __launch_bounds__(128) lnl_sum_finish_kernel(const double* __restrict__ P, int n, int ld,
                                                             const int32_t* __restrict__ n_dev,
                                                             const double* __restrict__ ws, int n_groups,
                                                             int log2_groups, double* __restrict__ out) {
  const int nv = n_dev ? min(n, *n_dev) : n;
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= nv) return;
  const double v = sum_groups(ws, n, c, n_groups, log2_groups, lane);
  if (lane == 0) {
    SumTheta th;
    th.load(P + (size_t)c * ld);
    out[c] = sum_finish_value(sum_prior(th.ptr()), v);
  }
}
#endif  // BPM_JIT_SUM

}  // namespace bpm

#if defined(BPM_JIT_SUM) && defined(BPM_JIT_PROBLEMS)
#include "cr_reduce.cuh"     // cr_update_problems_kernel
namespace bpm {
// Multi-problem handles (engine.cu: kJitSumProblems): data is [BPM_NPROBLEMS][BPM_NROWS][BPM_ROWLEN], and rows
// [g rpp, (g + 1) rpp) of P belong to problem g.  The body of lnl_sum_kernel on a tile that never straddles two
// problems: block x holds tile x % tpp (tpp = ceil(rpp / tile)) of problem g = x / tpp and reads problem g's rows, so
// every sum is added in the order of one problem of M rows.  A phase's idle slot (n odd: the last of the smaller
// half) is evaluated like the others on whatever proposal row it holds; accept never reads its result.
// grid (P tpp, n_groups), kSumThreads threads; dynamic shared memory sum_smem_bytes(tile).
__global__ void __launch_bounds__(kSumThreads) lnl_sum_problems_kernel(const double* __restrict__ P, int n, int ld,
                                                                       int rpp, int tpp,
                                                                       const double* __restrict__ data, int tile,
                                                                       int log2_group, int n_groups,
                                                                       double* __restrict__ ws,
                                                                       double* __restrict__ out) {
  extern __shared__ __align__(16) double sm_sum[];
  const int g = blockIdx.x / tpp;
  const int t0 = (blockIdx.x - g * tpp) * tile;         // first row of the tile inside problem g
  const int c0 = g * rpp + t0;
  const int nt = min(tile, rpp - t0);
  const double* __restrict__ pdata = data + (int64_t)g * kSumRows * kSumK;
  double* stk = sm_sum;                                  // [tile][kSumMaxDepth]
  double* prior = stk + tile * kSumMaxDepth;             // [tile]
  double* srows = prior + tile;                          // [k][kSumStageRows] when staged
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t G = (int64_t)1 << log2_group;
  const int64_t q0 = (int64_t)blockIdx.y * G;
  for (int ci = threadIdx.x; ci < nt; ci += kSumThreads) {
    SumTheta th;
    th.load(P + (size_t)(c0 + ci) * ld);
    prior[ci] = sum_prior(th.ptr());
  }
  __syncthreads();
  const int64_t m = min(G, kSumChunks - q0);
  const int sc = G < kSumStageChunks ? (int)G : kSumStageChunks;
  for (int64_t s0 = 0; s0 < m; s0 += sc) {
    const int64_t r0 = (q0 + s0) * kSumChunk;
    const int ns = (int)min((int64_t)sc, m - s0);
    if constexpr (kSumStaged) {
      __syncthreads();
      sum_stage(srows, pdata, r0, min((int64_t)ns * kSumChunk, kSumRows - r0));
      __syncthreads();
    }
    for (int ci = warp; ci < nt; ci += kSumThreads / 32) {
      if (prior[ci] == -INFINITY) continue;
      double* cs = stk + ci * kSumMaxDepth;
      SumTheta th;
      th.load(P + (size_t)(c0 + ci) * ld);
      for (int s = 0; s < ns; ++s)
        sum_push(cs, s0 + s, sum_chunk(th.ptr(), q0 + s0 + s, srows, r0, pdata, kSumRows, lane), lane);
    }
  }
  __syncthreads();
  for (int ci = threadIdx.x; ci < nt; ci += kSumThreads) {
    const double S = sum_flush(stk + ci * kSumMaxDepth, m, log2_group);
    if (n_groups == 1) out[c0 + ci] = sum_finish_value(prior[ci], S);
    else ws[(size_t)blockIdx.y * n + c0 + ci] = S;
  }
}
}  // namespace bpm
#endif

#ifdef BPM_JIT_SUM_RAGGED
#include "cr_reduce.cuh"     // cr_update_problems_kernel (BPM_JIT_PROBLEMS is defined too)
namespace bpm {
// Multi-problem handles with datasets of different lengths (engine.cu: kJitSumRagged).  data is the concatenated
// [sum_g M_g][BPM_ROWLEN] array, problem g's M_g rows start at row row_off[g] (row_off[BPM_NPROBLEMS] = sum_g M_g),
// and rows [g rpp, (g + 1) rpp) of P belong to problem g.  Problem g's tree has C_g = ceil(M_g / 256) chunks and
// P2_g leaves; it uses groups of G_g = min(G, P2_g) chunks, G = 2^log2_group the launch's, so a problem shorter
// than a group ends its tree at P2_g as a single-problem handle does (one more level of + 0.0 would turn a -0.0 sum
// into +0.0).
struct RaggedGroups {
  int64_t M;      // rows
  int64_t C;      // chunks
  int lg;         // log2(G_g)
  int n_groups;   // ceil(C / G_g)
  int log2_groups;// log2(P2_g / G_g)
  __device__ __forceinline__ RaggedGroups(const int64_t* __restrict__ row_off, int g, int log2_group) {
    M = row_off[g + 1] - row_off[g];
    C = (M + kSumChunk - 1) / kSumChunk;
    const int lp2 = C > 1 ? 64 - __clzll(C - 1) : 0;
    lg = min(log2_group, lp2);
    n_groups = (int)((C + ((int64_t)1 << lg) - 1) >> lg);
    log2_groups = lp2 - lg;
  }
};

// The body of lnl_sum_problems_kernel with problem g's row count taken at run time.  The grid is a flat work list:
// problem g owns blocks [blk_off[g], blk_off[g + 1]), tpp tiles (tpp = ceil(rpp / tile)) times its groups, tiles
// of one group adjacent.  A problem of one group writes ln L; otherwise group partials go to ws[ng_max][n] and
// lnl_sum_ragged_finish_kernel completes them.  kSumThreads threads; dynamic shared memory sum_smem_bytes(tile).
__global__ void __launch_bounds__(kSumThreads) lnl_sum_ragged_kernel(const double* __restrict__ P, int n, int ld,
                                                                     int rpp, int tpp,
                                                                     const double* __restrict__ data,
                                                                     const int64_t* __restrict__ row_off,
                                                                     const int32_t* __restrict__ blk_off, int tile,
                                                                     int log2_group, double* __restrict__ ws,
                                                                     double* __restrict__ out) {
  extern __shared__ __align__(16) double sm_sum[];
  const int b = blockIdx.x;
  int g = 0, hi = BPM_NPROBLEMS;                          // blk_off[g] <= b < blk_off[g + 1]
  while (hi - g > 1) {
    const int mid = (g + hi) >> 1;
    if (blk_off[mid] <= b) g = mid;
    else hi = mid;
  }
  const RaggedGroups pg(row_off, g, log2_group);
  const int local = b - blk_off[g];
  const int grp = local / tpp;
  const int t0 = (local - grp * tpp) * tile;             // first row of the tile inside problem g
  const int c0 = g * rpp + t0;
  const int nt = min(tile, rpp - t0);
  const double* __restrict__ pdata = data + row_off[g] * kSumK;
  double* stk = sm_sum;                                  // [tile][kSumMaxDepth]
  double* prior = stk + tile * kSumMaxDepth;             // [tile]
  double* srows = prior + tile;                          // [k][kSumStageRows] when staged
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t G = (int64_t)1 << pg.lg;
  const int64_t q0 = (int64_t)grp * G;
  for (int ci = threadIdx.x; ci < nt; ci += kSumThreads) {
    SumTheta th;
    th.load(P + (size_t)(c0 + ci) * ld);
    prior[ci] = sum_prior(th.ptr());
  }
  __syncthreads();
  const int64_t m = min(G, pg.C - q0);
  const int sc = G < kSumStageChunks ? (int)G : kSumStageChunks;
  for (int64_t s0 = 0; s0 < m; s0 += sc) {
    const int64_t r0 = (q0 + s0) * kSumChunk;
    const int ns = (int)min((int64_t)sc, m - s0);
    if constexpr (kSumStaged) {
      __syncthreads();
      sum_stage(srows, pdata, r0, min((int64_t)ns * kSumChunk, pg.M - r0));
      __syncthreads();
    }
    for (int ci = warp; ci < nt; ci += kSumThreads / 32) {
      if (prior[ci] == -INFINITY) continue;
      double* cs = stk + ci * kSumMaxDepth;
      SumTheta th;
      th.load(P + (size_t)(c0 + ci) * ld);
      for (int s = 0; s < ns; ++s)
        sum_push(cs, s0 + s, sum_chunk(th.ptr(), q0 + s0 + s, srows, r0, pdata, pg.M, lane), lane);
    }
  }
  __syncthreads();
  for (int ci = threadIdx.x; ci < nt; ci += kSumThreads) {
    const double S = sum_flush(stk + ci * kSumMaxDepth, m, pg.lg);
    if (pg.n_groups == 1) out[c0 + ci] = sum_finish_value(prior[ci], S);
    else ws[(size_t)grp * n + c0 + ci] = S;
  }
}

// Step 3 above the groups and step 4 for the rows of problems of several groups, one warp per row (sum_groups over
// the problem's own n_groups and log2_groups); rows of one-group problems were written by the sum kernel.
__global__ void __launch_bounds__(128) lnl_sum_ragged_finish_kernel(const double* __restrict__ P, int n, int ld,
                                                                    int rpp, const int64_t* __restrict__ row_off,
                                                                    const double* __restrict__ ws, int log2_group,
                                                                    double* __restrict__ out) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= n) return;
  const RaggedGroups pg(row_off, c / rpp, log2_group);
  if (pg.n_groups == 1) return;
  const double v = sum_groups(ws, n, c, pg.n_groups, pg.log2_groups, lane);
  if (lane == 0) {
    SumTheta th;
    th.load(P + (size_t)c * ld);
    out[c] = sum_finish_value(sum_prior(th.ptr()), v);
  }
}
}  // namespace bpm
#endif  // BPM_JIT_SUM_RAGGED
