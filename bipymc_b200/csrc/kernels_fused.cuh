// Fused half-phase kernels: RNG + proposal + likelihood + Metropolis accept + in-place
// state / moments / history update in ONE launch (demc.py:153-196, dream.py:32-107 for a
// whole half of the population).
//
// Correlated-Gaussian target, 5 <= d <= 108 (the 100-D headline case), one persistent
// warp-specialised CTA per SM: producer warps draw, gather and build the proposals of a
// 64-chain tile, consumer warps run the quadratic form and the Metropolis decision.
// gauss_fused_kernel (end of this file) picks the kernel from the shape:
//  * fused_gauss_v4_kernel (kernels_fused_v4.cuh) -- the default: partner rows staged in
//    shared memory by TMA, quadratic form on the FP64 tensor pipe (DMMA), lazy history /
//    moments protocol (PhaseArgs::pending).  Needs d % 4 == 0, ld == d and its landing
//    slots to fit shared memory.
//  * fused_gauss_v3_kernel -- the same pipeline with register gathers, where v4's landing
//    slots do not fit (larger d or more pairs), and on request (BPM_FUSED_GAUSS_V3).
//  * fused_gauss_ws_kernel -- 12 producer / 8 DFMA consumer warps, eager write-back, where
//    v3 / v4 cannot run (d % 4 != 0 or ld != d), and on request (BPM_FUSED_GAUSS_WS).
// d <= 4 analytic targets (banana, bimodal, line fit): fused_small_kernel, thread per
// chain (kernels_small.cuh, which the run-time compiled likelihoods share).
// All of them share every draw / arithmetic helper with the generic split path (step.cuh),
// so the chains they produce are bit-identical to it.
#pragma once
#include <cuda_runtime.h>
#include "step.cuh"
#include "targets.cuh"
#include "kernels_small.cuh"

namespace bpm {

constexpr int kTileRows = 64;    // chains per tile
constexpr int kColStrip = 14;    // columns per warp in the quadratic form
constexpr int kWld = 8 * kColStrip;  // padded row length of W in shared memory (112)
constexpr int kHalfThreads = 256;

// Row sums of squares of (P - mu) . W for a 64-row tile held in shared memory.
//   P     [64][pld]   row-major, pld odd (conflict-free column walks)
//   Ws    [d][112]    zero-padded columns
//   part  [8][64]     per-warp partial sums, summed in warp order by the caller
// 256 threads: lane = row (and row + 32), warp = 14-column strip.
template <bool CENTER>
__device__ __forceinline__ void gauss_tile_rowsums(const double* __restrict__ P, int pld,
                                                   const double* __restrict__ Ws,
                                                   const double* __restrict__ mus, int d,
                                                   double* __restrict__ part, int warp, int lane) {
  double a0[kColStrip], a1[kColStrip];
#pragma unroll
  for (int q = 0; q < kColStrip; ++q) a0[q] = a1[q] = 0.0;
  const double* p0 = P + lane * pld;
  const double* p1 = P + (lane + 32) * pld;
  const double2* wv = reinterpret_cast<const double2*>(Ws + warp * kColStrip);
#pragma unroll 2
  for (int k = 0; k < d; ++k) {
    double x0 = p0[k], x1 = p1[k];
    if (CENTER) {
      const double m = mus[k];
      x0 = __dsub_rn(x0, m);
      x1 = __dsub_rn(x1, m);
    }
#pragma unroll
    for (int q = 0; q < kColStrip / 2; ++q) {
      const double2 b = wv[k * (kWld / 2) + q];
      a0[2 * q] = fma(x0, b.x, a0[2 * q]);
      a0[2 * q + 1] = fma(x0, b.y, a0[2 * q + 1]);
      a1[2 * q] = fma(x1, b.x, a1[2 * q]);
      a1[2 * q + 1] = fma(x1, b.y, a1[2 * q + 1]);
    }
  }
  double s0 = 0.0, s1 = 0.0;
#pragma unroll
  for (int q = 0; q < kColStrip; ++q) {
    s0 = fma(a0[q], a0[q], s0);
    s1 = fma(a1[q], a1[q], s1);
  }
  part[warp * kTileRows + lane] = s0;
  part[warp * kTileRows + lane + 32] = s1;
}

__device__ __forceinline__ double gauss_tile_finish(const double* __restrict__ part, int row, double c0,
                                                    int log_of_pdf) {
  double maha = part[row];
#pragma unroll
  for (int w = 1; w < 8; ++w) maha = __dadd_rn(maha, part[w * kTileRows + row]);
  return gauss_finish(c0, maha, log_of_pdf);
}

__device__ __forceinline__ void load_W_shared(double* Ws, double* mus, const double* __restrict__ W,
                                              const double* __restrict__ mu, int d, int r, int tid,
                                              int nthreads) {
  for (int idx = tid; idx < d * kWld; idx += nthreads) {
    const int k = idx / kWld, j = idx - k * kWld;
    Ws[idx] = j < r ? W[(size_t)k * r + j] : 0.0;
  }
  for (int k = tid; k < d; k += nthreads) mus[k] = mu[k];
}

inline bool gauss_rows_supported(int d, int r) { return d <= 112 && r <= kWld && d >= 5; }
constexpr size_t kMaxDynSmem = 232448;   // opt-in dynamic shared memory per CTA on sm_100
inline int gauss_pld(int d) { return d | 1; }

// ---- stand-alone batched likelihood with the same tile arithmetic ------------------
template <bool CENTER>
__global__ void __launch_bounds__(kHalfThreads, 1)
gauss_rows_kernel(const double* __restrict__ X, int n, int ld, int d, int r, const double* __restrict__ mu,
                  const double* __restrict__ W, double c0, int log_of_pdf, double* __restrict__ out) {
  extern __shared__ __align__(16) double smem[];
  const int pld = d | 1;
  double* Ws = smem;
  double* mus = Ws + d * kWld;
  double* P = mus + ((d + 1) & ~1);
  double* part = P + kTileRows * pld;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  load_W_shared(Ws, mus, W, mu, d, r, threadIdx.x, kHalfThreads);
  const int n_tiles = (n + kTileRows - 1) / kTileRows;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    __syncthreads();
    for (int idx = threadIdx.x; idx < kTileRows * d; idx += kHalfThreads) {
      const int rr = idx / d, k = idx - rr * d;
      const int row = tile * kTileRows + rr;
      P[rr * pld + k] = row < n ? X[(size_t)row * ld + k] : 0.0;
    }
    __syncthreads();
    gauss_tile_rowsums<CENTER>(P, pld, Ws, mus, d, part, warp, lane);
    __syncthreads();
    if (threadIdx.x < kTileRows) {
      const int row = tile * kTileRows + threadIdx.x;
      if (row < n) out[row] = gauss_tile_finish(part, threadIdx.x, c0, log_of_pdf);
    }
  }
}

inline size_t gauss_rows_smem(int d) {
  return sizeof(double) * ((size_t)d * kWld + ((d + 1) & ~1) + (size_t)kTileRows * gauss_pld(d) +
                           8 * kTileRows);
}

inline int launch_gauss_rows(const double* X, int n, int ld, int d, int r, const double* mu,
                             const double* W, double c0, int log_of_pdf, int mu_is_zero, double* out,
                             cudaStream_t s) {
  const size_t sm = gauss_rows_smem(d);
  const int n_tiles = (n + kTileRows - 1) / kTileRows;
  const int grid = n_tiles < 148 ? n_tiles : 148;
  cudaError_t e;
  if (mu_is_zero) {
    e = cudaFuncSetAttribute(gauss_rows_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    if (e != cudaSuccess) return 1;
    gauss_rows_kernel<false><<<grid, kHalfThreads, sm, s>>>(X, n, ld, d, r, mu, W, c0, log_of_pdf, out);
  } else {
    e = cudaFuncSetAttribute(gauss_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    if (e != cudaSuccess) return 1;
    gauss_rows_kernel<true><<<grid, kHalfThreads, sm, s>>>(X, n, ld, d, r, mu, W, c0, log_of_pdf, out);
  }
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

// ---- the fused Gaussian half-phase ----------------------------------------------------
struct GaussArgs {
  const double* mu;
  const double* W;
  const double* Wf;   // W in DMMA fragment order (w_fragment_kernel, built once per bpm_set_target), or nullptr
  int r;
  double c0;
  int log_of_pdf;
};

// Shared-memory scratch of one 64-chain tile.
struct TileScratch {
  double gamma_u[kTileRows];
  double accept_u[kTileRows];
  int cid[kTileRows];           // global chain id, -1 = empty row
  int cr_idx[kTileRows];
  int fallback[kTileRows];
  int acc[kTileRows];
  int pa[kTileRows][BPM_MAX_PAIRS];   // GLOBAL chain ids of the partner rows
  int pb[kTileRows][BPM_MAX_PAIRS];
};

// Kernel-lifetime tables in shared memory.
struct GaussTables {
  double* Ws;    // [d][112] whitening matrix, zero-padded columns
  double* mus;   // [d]
  double* gam;   // gamma_base[d'] for d' = 0..d (dream.py:61)
  double* cdf;   // normalised CR cdf (dream.py:51)
  double* crv;   // CR values (dream.py:113)
  uint32_t* thr; // native mode: mask_i = (12-bit z word <= thr[m])  <=>  z_i <= CR[m]   (zen_threshold)
};
__host__ __device__ inline size_t gauss_table_doubles(int d) {
  return (size_t)d * kWld + ((d + 1) & ~1) + ((d + 2) & ~1) + 2 * BPM_MAX_CR + BPM_MAX_CR / 2;
}
// one proposal tile: P[64][pld] followed by the consumers' partial sums part[8][64]
__host__ __device__ inline size_t gauss_ptile_doubles(int d) {
  return (((size_t)kTileRows * (d | 1) + 1) & ~(size_t)1) + 8 * kTileRows;
}
__host__ __device__ inline size_t gauss_scratch_doubles() { return (sizeof(TileScratch) + 7) / 8; }

__device__ __forceinline__ GaussTables carve_tables(double* smem, int d) {
  GaussTables t;
  t.Ws = smem;
  t.mus = t.Ws + d * kWld;
  t.gam = t.mus + ((d + 1) & ~1);
  t.cdf = t.gam + ((d + 2) & ~1);
  t.crv = t.cdf + BPM_MAX_CR;
  t.thr = reinterpret_cast<uint32_t*>(t.crv + BPM_MAX_CR);
  return t;
}

// the small proposal-stage tables; the v3 / v4 kernels call this alone: their consumers load W (83 KB), in the
// shadow of the producers' first tile
__device__ __forceinline__ void fill_tables_v3(const PhaseArgs& a, const GaussArgs& g, const GaussTables& t,
                                               int tid, int nthreads) {
  for (int dp = tid; dp <= a.d; dp += nthreads)
    t.gam[dp] = dp == 0 ? 0.0
                        : __ddiv_rn(a.gamma_num, __dsqrt_rn(__dmul_rn(__dmul_rn(2.0, (double)a.del_pairs),
                                                                      (double)dp)));
  if (tid == 0) {
    double tot = 0.0;
    for (int m = 0; m < a.n_cr; ++m) tot = __dadd_rn(tot, a.p_cr[m]);
    double acc = 0.0;
    for (int m = 0; m < a.n_cr; ++m) {
      acc = __dadd_rn(acc, a.p_cr[m]);
      t.cdf[m] = __ddiv_rn(acc, tot);
      t.crv[m] = __ddiv_rn((double)(m + 1), (double)a.n_cr);
      t.thr[m] = zen_threshold(t.crv[m]);
    }
  }
}
__device__ __forceinline__ void fill_tables(const PhaseArgs& a, const GaussArgs& g, const GaussTables& t,
                                            int tid, int nthreads) {
  load_W_shared(t.Ws, t.mus, g.W, g.mu, a.d, g.r, tid, nthreads);
  fill_tables_v3(a, g, t, tid, nthreads);
}

// One instruction pulls a whole row into L2 (no registers, no shared memory): issued for
// every row a tile will touch, one pipeline step ahead of its use.
__device__ __forceinline__ void l2_prefetch_row(const double* p, int bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
// Streaming (evict-first) access for arrays that are touched once per generation -- running
// moments and history -- so they do not push the randomly gathered population out of L2.
__device__ __forceinline__ double2 ld_stream2(const double* p) {
  return __ldcs(reinterpret_cast<const double2*>(p));
}
__device__ __forceinline__ void st_stream2(double* p, double x, double y) {
  __stcs(reinterpret_cast<double2*>(p), make_double2(x, y));
}

// stage D: per-chain scalar draws, one thread per (chain, slot)
template <bool REPLAY>
__device__ __forceinline__ void tile_stage_draws(const PhaseArgs& a, const PhaseLists& L,
                                                 const GaussTables& tb, TileScratch& T, int tile,
                                                 int gtid, int gthreads) {
  const bool dream = a.algo == BPM_ALGO_DREAM;
  const int npair = dream ? a.del_pairs : 1;
  const int nslots = 2 + npair;
  for (int idx = gtid; idx < kTileRows * nslots; idx += gthreads) {
    const int row = idx / nslots, slot = idx - row * nslots;
    const int gid = tile * kTileRows + row;
    bool valid = gid < L.n_self;
    const int c = valid ? L.self[gid] : 0;
    valid = valid && c >= a.chain_lo && c < a.chain_hi;
    if (slot == 0) T.cid[row] = valid ? c : -1;
    if (!valid) continue;
    const int row_bytes = a.ld * 8;
    if (slot == 0) {
      l2_prefetch_row(a.X + (size_t)c * a.ld, row_bytes);
      if (a.mean) l2_prefetch_row(a.mean + (size_t)(c - a.chain_lo) * a.ld, row_bytes);
    } else if (slot == 1) {
      if (a.m2) l2_prefetch_row(a.m2 + (size_t)(c - a.chain_lo) * a.ld, row_bytes);
    }
    if (REPLAY) {
      if (slot == 0) {
        T.cr_idx[row] = dream ? a.rp.cr_idx[c] : 0;
        T.accept_u[row] = a.rp.accept_u[c];
      } else if (slot == 1) {
        T.gamma_u[row] = a.rp.gamma_u[c];
        T.fallback[row] = dream ? a.rp.fallback_dim[c] : -1;
      } else {
        const int p = slot - 2;
        T.pa[row][p] = L.pool[a.rp.pairs[((size_t)c * npair + p) * 2 + 0]];
        T.pb[row][p] = L.pool[a.rp.pairs[((size_t)c * npair + p) * 2 + 1]];
        l2_prefetch_row(a.X + (size_t)T.pa[row][p] * a.ld, row_bytes);
        l2_prefetch_row(a.X + (size_t)T.pb[row][p] * a.ld, row_bytes);
      }
    } else {
      const Philox4 q = draw4(a.rng, (uint32_t)c, RNG_SCALAR, (uint32_t)slot);
      if (slot == 0) {
        int m = 0;
        if (dream) {
          const double u = slot0_cr_u(q);
          for (int j = 0; j < a.n_cr; ++j)
            if (tb.cdf[j] <= u) m = j + 1;
          m = m < a.n_cr ? m : a.n_cr - 1;
        }
        T.cr_idx[row] = m;
        T.accept_u[row] = slot0_accept_u(q);
      } else if (slot == 1) {
        T.gamma_u[row] = slot1_gamma_u(q);
        T.fallback[row] = slot1_fallback(q, a.d);
      } else {
        int r1, r2;
        slot_pair(q, L.n_pool, r1, r2);
        const int ga = L.pool[r1], gb = L.pool[r2];
        T.pa[row][slot - 2] = ga;
        T.pb[row][slot - 2] = gb;
        l2_prefetch_row(a.X + (size_t)ga * a.ld, row_bytes);
        l2_prefetch_row(a.X + (size_t)gb * a.ld, row_bytes);
      }
    }
  }
}

// stage A: crossover mask, row gathers, proposal -> P tile (a warp per chain row)
template <bool REPLAY>
__device__ __forceinline__ void tile_stage_propose(const PhaseArgs& a, const GaussTables& tb,
                                                   TileScratch& T, double* __restrict__ P, int pld,
                                                   int gwarp, int gwarps, int lane) {
  const int d = a.d;
  const bool dream = a.algo == BPM_ALGO_DREAM;
  const int npair = dream ? a.del_pairs : 1;
  const int blk = lane;                  // this lane's dimension block (4 doubles)
  const bool has_blk = 4 * blk < d;
  const bool full = 4 * blk + 3 < d;
  for (int row = gwarp; row < kTileRows; row += gwarps) {
    const int c = T.cid[row];
    double* prow = P + row * pld;
    if (c < 0) {
      if (has_blk)
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (4 * blk + q < d) prow[4 * blk + q] = 0.0;
      continue;
    }
    // issue the row gathers first: they do not depend on the mask draws
    double cur[4] = {0, 0, 0, 0}, S[4] = {0, 0, 0, 0}, var[4] = {0, 0, 0, 0};
    const bool welford_var = dream && a.adapt && !(REPLAY && a.hist_base != nullptr);
    if (has_blk) {
      const double* xc = a.X + (size_t)c * a.ld + 4 * blk;
      if (welford_var) {   // same arithmetic as cr_variance(), loads issued with the gathers
        const double* mp = a.m2 + (size_t)(c - a.chain_lo) * a.ld + 4 * blk;
        if (full) {
          const double2 w0 = ld_stream2(mp), w1 = ld_stream2(mp + 2);
          var[0] = w0.x; var[1] = w0.y; var[2] = w1.x; var[3] = w1.y;
        } else {
#pragma unroll
          for (int q = 0; q < 4; ++q) var[q] = 4 * blk + q < d ? mp[q] : 0.0;
        }
      }
      if (full) {
        const double2 u0 = *reinterpret_cast<const double2*>(xc);
        const double2 u1 = *reinterpret_cast<const double2*>(xc + 2);
        cur[0] = u0.x; cur[1] = u0.y; cur[2] = u1.x; cur[3] = u1.y;
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) cur[q] = 4 * blk + q < d ? xc[q] : 0.0;
      }
#pragma unroll
      for (int p = 0; p < BPM_MAX_PAIRS; ++p) {
        if (p < npair) {
          const double* pa = a.X + (size_t)T.pa[row][p] * a.ld + 4 * blk;
          const double* pb = a.X + (size_t)T.pb[row][p] * a.ld + 4 * blk;
          double va[4], vb[4];
          if (full) {
            const double2 s0 = *reinterpret_cast<const double2*>(pa);
            const double2 s1 = *reinterpret_cast<const double2*>(pa + 2);
            const double2 t0 = *reinterpret_cast<const double2*>(pb);
            const double2 t1 = *reinterpret_cast<const double2*>(pb + 2);
            va[0] = s0.x; va[1] = s0.y; va[2] = s1.x; va[3] = s1.y;
            vb[0] = t0.x; vb[1] = t0.y; vb[2] = t1.x; vb[3] = t1.y;
          } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              va[q] = 4 * blk + q < d ? pa[q] : 0.0;
              vb[q] = 4 * blk + q < d ? pb[q] : 0.0;
            }
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const double df = __dsub_rn(va[q], vb[q]);
            S[q] = p == 0 ? df : __dadd_rn(S[q], df);
          }
        }
      }
    }
    uint32_t mbits = 0xFu;
    double gamma;
    const double gu = T.gamma_u[row];
    if (dream) {
      mbits = 0u;
      const double cr = tb.crv[T.cr_idx[row]];
      if (has_blk) {
        double z[4];
        z4<REPLAY>(a, c, blk, z);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (4 * blk + q < d && z[q] <= cr) mbits |= 1u << q;
      }
      int d_prime = __reduce_add_sync(0xFFFFFFFFu, __popc(mbits));
      if (d_prime == 0) {
        const int fb = T.fallback[row] < 0 ? 0 : T.fallback[row];
        if ((fb >> 2) == blk) mbits |= 1u << (fb & 3);
        d_prime = 1;
      }
      gamma = tb.gam[d_prime];
      if (a.gamma_jump) gamma = gu < a.gamma_p0 ? gamma : 1.0;
    } else {
      gamma = demc_gamma(a, gu);
    }
    double delta = 0.0;
    if (has_blk) {
      double e[4], nn[4];
      en4<REPLAY>(a, c, blk, e, nn);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i = 4 * blk + q;
        if (i < d) {
          double pr;
          if (dream) {
            pr = dream_prop(cur[q], S[q], e[q], nn[q], gamma, (mbits >> q) & 1u ? 1.0 : 0.0);
            if (a.adapt) {
              double v;
              if (welford_var) {
                v = __dmul_rn(var[q], a.inv_mom);
                if (!(v > 0.0)) v = 1e-12 * 1e-12;
              } else {
                v = cr_variance<REPLAY>(a, c, i);
              }
              delta += cr_term(cur[q], pr, v);
            }
          } else {
            pr = demc_prop(cur[q], S[q], nn[q], gamma);
          }
          prow[i] = pr;
          if (REPLAY && a.tr.prop) a.tr.prop[(size_t)c * d + i] = pr;
        }
      }
    }
    if (dream) {
      delta = group_sum_d<32>(delta);
      if (lane == 0) {
        a.cr_pick[c] = a.adapt ? T.cr_idx[row] : -1;
        a.cr_delta[c] = delta;
      }
    }
  }
}

// after stage B: likelihood value + Metropolis decision of chain row `row` (one thread each);
// must be called by whole warps (ballots).  Adds to the caller's accept / reject tallies.
__device__ __forceinline__ void tile_stage_decide(const PhaseArgs& a, const GaussArgs& g, TileScratch& T,
                                                  const double* __restrict__ part, int row,
                                                  unsigned& n_acc, unsigned& n_rej) {
  const int c = T.cid[row];
  int acc = 0;
  if (c >= 0) {
    const double lp = gauss_tile_finish(part, row, g.c0, g.log_of_pdf);
    acc = metropolis(a.lnl[c], lp, T.accept_u[row]);
    if (acc < 0) {
      *a.nan_flag = 1;
      acc = 0;
    }
    if (acc) a.lnl[c] = lp;
    if (a.tr.accept) a.tr.accept[c] = acc;
    if (a.tr.lnl_prop) a.tr.lnl_prop[c] = lp;
  }
  T.acc[row] = acc;
  n_acc += __popc(__ballot_sync(0xFFFFFFFFu, c >= 0 && acc));
  n_rej += __popc(__ballot_sync(0xFFFFFFFFu, c >= 0 && !acc));
}

// stage C: the single write-back (state, running moments, history row)
__device__ __forceinline__ void tile_stage_writeback(const PhaseArgs& a, const TileScratch& T,
                                                     const double* __restrict__ P, int pld, int gwarp,
                                                     int gwarps, int lane) {
  const int d = a.d;
  const int blk = lane;
  if (4 * blk >= d) return;
  const bool full = 4 * blk + 3 < d;
  for (int row = gwarp; row < kTileRows; row += gwarps) {
    const int c = T.cid[row];
    if (c < 0) continue;
    const int acc = T.acc[row];
    double* xc = a.X + (size_t)c * a.ld + 4 * blk;
    const double* prow = P + row * pld + 4 * blk;
    const size_t o = (size_t)(c - a.chain_lo) * a.ld + 4 * blk;
    double s[4] = {0, 0, 0, 0};
    if (acc) {
#pragma unroll
      for (int q = 0; q < 4; ++q) s[q] = 4 * blk + q < d ? prow[q] : 0.0;
      if (full) {
        *reinterpret_cast<double2*>(xc) = make_double2(s[0], s[1]);
        *reinterpret_cast<double2*>(xc + 2) = make_double2(s[2], s[3]);
        store_peers4(a, (size_t)c * a.ld + 4 * blk, s[0], s[1], s[2], s[3]);
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (4 * blk + q < d) {
            xc[q] = s[q];
            store_peers1(a, (size_t)c * a.ld + 4 * blk + q, s[q]);
          }
      }
    } else if (a.mean || a.hist_row) {
      if (full) {
        const double2 u0 = *reinterpret_cast<const double2*>(xc);
        const double2 u1 = *reinterpret_cast<const double2*>(xc + 2);
        s[0] = u0.x; s[1] = u0.y; s[2] = u1.x; s[3] = u1.y;
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) s[q] = 4 * blk + q < d ? xc[q] : 0.0;
      }
    }
    if (a.mean) {
      if (full) {
        double2 m0 = ld_stream2(a.mean + o), m1 = ld_stream2(a.mean + o + 2);
        double2 v0 = ld_stream2(a.m2 + o), v1 = ld_stream2(a.m2 + o + 2);
        welford_update(s[0], a.inv_n1, m0.x, v0.x);
        welford_update(s[1], a.inv_n1, m0.y, v0.y);
        welford_update(s[2], a.inv_n1, m1.x, v1.x);
        welford_update(s[3], a.inv_n1, m1.y, v1.y);
        st_stream2(a.mean + o, m0.x, m0.y);
        st_stream2(a.mean + o + 2, m1.x, m1.y);
        st_stream2(a.m2 + o, v0.x, v0.y);
        st_stream2(a.m2 + o + 2, v1.x, v1.y);
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (4 * blk + q < d) {
            double mu = a.mean[o + q], v = a.m2[o + q];
            welford_update(s[q], a.inv_n1, mu, v);
            a.mean[o + q] = mu;
            a.m2[o + q] = v;
          }
      }
    }
    if (a.hist_row) {
      if (full) {
        st_stream2(a.hist_row + o, s[0], s[1]);
        st_stream2(a.hist_row + o + 2, s[2], s[3]);
      } else {
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (4 * blk + q < d) a.hist_row[o + q] = s[q];
      }
    }
  }
}

// shared memory of fused_gauss_ws_kernel: tables, 2 proposal tiles, 3 scratch blocks
inline size_t fused_gauss_smem(int d) {
  return sizeof(double) * (gauss_table_doubles(d) + 2 * gauss_ptile_doubles(d) + 3 * gauss_scratch_doubles());
}

// fused_gauss_ws_kernel: warp-specialised producer / consumer pipeline.
//   8 consumer warps (128 registers each) run nothing but the FP64 tile GEMM + the
//   Metropolis decision; 12 producer warps (72 registers each) run the latency-bound
//   stages -- draws, row gathers, proposal, write-back.  Two tile buffers rotate between
//   the groups through named barriers (FULL[b]: producers -> consumers, DONE[b]: back), so
//   the FP64 pipe works on tile i while the producers finalise tile i-1 and gather tile
//   i+1.  setmaxnreg moves registers from the producer to the consumer warpgroups.
constexpr int kConsWarps = 8, kProdWarps = 12;
constexpr int kWsThreads = 32 * (kConsWarps + kProdWarps);   // 640
constexpr int kProdThreads = 32 * kProdWarps;
constexpr int kConsThreads = 32 * kConsWarps;
enum { BAR_PROD = 1, BAR_CONS = 2, BAR_FULL0 = 3, BAR_FULL1 = 4, BAR_DONE0 = 5, BAR_DONE1 = 6 };

__device__ __forceinline__ void nbar_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void nbar_arrive(int id, int count) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory");
}

template <bool REPLAY, bool CENTER>
__global__ void __launch_bounds__(kWsThreads, 1)
fused_gauss_ws_kernel(const PhaseArgs a, const GaussArgs g) {
  extern __shared__ __align__(16) double smem[];
  const int d = a.d, pld = d | 1;
  const GaussTables tb = carve_tables(smem, d);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* Pbuf = smem + gauss_table_doubles(d);
  const size_t p_stride = gauss_ptile_doubles(d);
  const size_t part_off = ((size_t)kTileRows * pld + 1) & ~(size_t)1;
  double* Tbuf = Pbuf + 2 * p_stride;
  const size_t t_stride = gauss_scratch_doubles();
  fill_tables(a, g, tb, threadIdx.x, kWsThreads);
  __syncthreads();
  const PhaseLists L = phase_lists(a);
  const int n_tiles = (L.n_self + kTileRows - 1) / kTileRows;
  const int n_my = blockIdx.x < n_tiles ? (n_tiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;

  if (warp < kConsWarps) {
    // ------------------------------ consumers ------------------------------------------
    asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
    unsigned n_acc = 0, n_rej = 0;
    for (int i = 0; i < n_my; ++i) {
      const int b = i & 1;
      double* P = Pbuf + b * p_stride;
      double* part = P + part_off;
      TileScratch& T = *reinterpret_cast<TileScratch*>(Tbuf + (i % 3) * t_stride);
      nbar_sync(BAR_FULL0 + b, kWsThreads);            // producers filled buffer b
      gauss_tile_rowsums<CENTER>(P, pld, tb.Ws, tb.mus, d, part, warp, lane);
      nbar_sync(BAR_CONS, kConsThreads);
      if (threadIdx.x < kTileRows) tile_stage_decide(a, g, T, part, threadIdx.x, n_acc, n_rej);
      nbar_arrive(BAR_DONE0 + b, kWsThreads);          // decisions of tile i are in T.acc
    }
    if (lane == 0) {
      if (n_acc) atomicAdd(a.n_acc, (unsigned long long)n_acc);
      if (n_rej) atomicAdd(a.n_rej, (unsigned long long)n_rej);
    }
  } else {
    // ------------------------------ producers ------------------------------------------
    // software pipeline, one iteration = draws + L2 prefetch of tile i+1 | proposal of
    // tile i | write-back of tile i-1
    asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
    const int pw = warp - kConsWarps;
    const int ptid = threadIdx.x - kConsThreads;
    if (n_my > 0)
      tile_stage_draws<REPLAY>(a, L, tb, *reinterpret_cast<TileScratch*>(Tbuf), blockIdx.x, ptid,
                               kProdThreads);
    nbar_sync(BAR_PROD, kProdThreads);
    for (int i = 0; i <= n_my; ++i) {
      if (i + 1 < n_my)
        tile_stage_draws<REPLAY>(a, L, tb, *reinterpret_cast<TileScratch*>(Tbuf + ((i + 1) % 3) * t_stride),
                                 blockIdx.x + (i + 1) * gridDim.x, ptid, kProdThreads);
      if (i < n_my) {
        const int b = i & 1;
        double* P = Pbuf + b * p_stride;
        TileScratch& T = *reinterpret_cast<TileScratch*>(Tbuf + (i % 3) * t_stride);
        tile_stage_propose<REPLAY>(a, tb, T, P, pld, pw, kProdWarps, lane);
        nbar_arrive(BAR_FULL0 + b, kWsThreads);
      }
      if (i >= 1) {
        const int b2 = (i - 1) & 1;
        const double* P = Pbuf + b2 * p_stride;
        const TileScratch& T = *reinterpret_cast<const TileScratch*>(Tbuf + ((i - 1) % 3) * t_stride);
        nbar_sync(BAR_DONE0 + b2, kWsThreads);          // consumers decided tile i-1
        tile_stage_writeback(a, T, P, pld, pw, kProdWarps, lane);
      }
      // draws of tile i+1 are complete and buffers of tile i-1 are free for every producer
      nbar_sync(BAR_PROD, kProdThreads);
    }
  }
}


// ---- FP64 tensor-core (DMMA) tile product for variant 3 -------------------------------
// B200 measures the same FP64 peak through mma.sync.m8n8k4.f64 as through DFMA
// (profiles/r1_fp64_probe_b200.txt), but one DMMA replaces eight DFMA warp instructions
// and its operand fragments are 1 double per lane, so the consumer needs ~10x less
// shared-memory return bandwidth than the register-tiled DFMA form (which profiling
// showed to be LSU-bound: 256 LSU cycles against 112 FP64 cycles per k step).
//   A fragment (8 x 4, row): lane l holds A[l / 4][l % 4]       <- proposal tile P
//   B fragment (4 x 8, col): lane l holds B[l % 4][l / 4]       <- W, stored in fragment order
//   C fragment (8 x 8):      lane l holds C[l / 4][2 (l % 4) + {0, 1}]
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__host__ __device__ inline int dmma_pld(int d) {          // row stride = 4 or 12 (mod 16) doubles:
  int p = d;                                              // conflict-free A-fragment loads
  while ((p & 15) != 4 && (p & 15) != 12) ++p;
  return p;
}
__host__ __device__ inline int dmma_ntiles(int r) { return (r + 7) >> 3; }
// Wf[(k4 * NT + nt) * 32 + lane] = W[4 k4 + lane % 4][8 nt + lane / 4]  (0 outside d x r)
__device__ __forceinline__ void load_W_fragments(double* Wf, double* mus, const double* __restrict__ W,
                                                 const double* __restrict__ mu, int d, int r, int tid,
                                                 int nthreads) {
  const int NT = dmma_ntiles(r);
  const int total = (d >> 2) * NT * 32;
  for (int idx = tid; idx < total; idx += nthreads) {
    const int lane = idx & 31, t = idx >> 5;
    const int k4 = t / NT, nt = t - k4 * NT;
    const int k = 4 * k4 + (lane & 3), j = 8 * nt + (lane >> 2);
    Wf[idx] = j < r ? W[(size_t)k * r + j] : 0.0;
  }
  for (int k = tid; k < d; k += nthreads) mus[k] = mu[k];
}

// The same layout written ONCE per target into global memory (bpm_set_target): the v4 kernel then brings W in
// with a single TMA bulk copy instead of 40 scattered loads + index divisions per consumer thread per launch.
__global__ void w_fragment_kernel(double* __restrict__ Wf, const double* __restrict__ W, int d, int r) {
  const int NT = dmma_ntiles(r);
  const int total = (d >> 2) * NT * 32;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int lane = idx & 31, t = idx >> 5;
    const int k4 = t / NT, nt = t - k4 * NT;
    const int k = 4 * k4 + (lane & 3), j = 8 * nt + (lane >> 2);
    Wf[idx] = j < r ? W[(size_t)k * r + j] : 0.0;
  }
}

// maha = |(P[row] - mu) . W|^2 for one m-tile (8 rows) per warp, no cross-warp hand-off: the four
// lanes of a quad end up holding the finished Mahalanobis distance of row 8 cw + lane / 4.
// A lone warp issues one DMMA.8x8x4 every ~50 cycles (profiles/r1_final_*: four consumer warps with
// 16 rows each were 90 % busy at a third of the FP64 tensor rate); two consumer warps per scheduler
// overlap each other's issue gaps (profiles/r1_consumer_experiments.txt).
template <bool CENTER>
__device__ __forceinline__ double gauss_tile_maha_dmma8(const double* __restrict__ P, int pld,
                                                        const double* __restrict__ Wf,
                                                        const double* __restrict__ mus, int d, int NT,
                                                        int cw, int lane) {
  const int r0 = 8 * cw + (lane >> 2), kq = lane & 3;
  const double* pa0 = P + r0 * pld + kq;
  const int nk4 = d >> 2;
  double s0 = 0.0;
  // column tiles in two groups of <= 7: 14 accumulators + the next k step's 7 B fragments fit the
  // 80 registers a consumer thread owns
#pragma unroll 1
  for (int g = 0; g < 2; ++g) {
    const int nt0 = 7 * g;
    const int cnt = NT - nt0 < 7 ? NT - nt0 : 7;
    if (cnt <= 0) break;
    double acc[7][2];
#pragma unroll
    for (int j = 0; j < 7; ++j) acc[j][0] = acc[j][1] = 0.0;
    const double* wf = Wf + nt0 * 32 + lane;
#pragma unroll 2
    for (int k4 = 0; k4 < nk4; ++k4) {
      double a0 = pa0[4 * k4];
      if (CENTER) a0 = __dsub_rn(a0, mus[4 * k4 + kq]);
      const double* wk = wf + (size_t)k4 * NT * 32;
#pragma unroll
      for (int j = 0; j < 7; ++j)
        if (j < cnt) dmma884(acc[j][0], acc[j][1], a0, wk[j * 32]);
    }
#pragma unroll
    for (int j = 0; j < 7; ++j)
      if (j < cnt) {
        s0 = fma(acc[j][0], acc[j][0], s0);
        s0 = fma(acc[j][1], acc[j][1], s0);
      }
  }
  s0 += __shfl_xor_sync(0xFFFFFFFFu, s0, 1);
  s0 += __shfl_xor_sync(0xFFFFFFFFu, s0, 2);
  return s0;
}

// Metropolis decision for one chain row whose Mahalanobis distance is in a register; called by whole
// warps, `row < 0` = this lane decides nothing.
__device__ __forceinline__ int tile_stage_decide_reg(const PhaseArgs& a, const GaussArgs& g, TileScratch& T,
                                                     double maha, int row, unsigned& n_acc, unsigned& n_rej) {
  const int c = row >= 0 ? T.cid[row] : -1;
  int acc = 0;
  if (c >= 0) {
    const double lp = gauss_finish(g.c0, maha, g.log_of_pdf);
    acc = metropolis(a.lnl[c], lp, T.accept_u[row]);
    if (acc < 0) {
      *a.nan_flag = 1;
      acc = 0;
    }
    if (acc) a.lnl[c] = lp;
    if (a.tr.accept) a.tr.accept[c] = acc;
    if (a.tr.lnl_prop) a.tr.lnl_prop[c] = lp;
  }
  if (row >= 0) T.acc[row] = acc;
  n_acc += __popc(__ballot_sync(0xFFFFFFFFu, c >= 0 && acc));
  n_rej += __popc(__ballot_sync(0xFFFFFFFFu, c >= 0 && !acc));
  return acc;
}

// =====================================================================================
// fused_gauss_v3_kernel: the same producer / consumer pipeline re-balanced after profiling
// fused_gauss_ws_kernel (profiles/r1_v2_*): its 8 consumer warps sat at the FULL barrier 76 % of the
// time while each of the 12 producer warps walked its chains serially at ~0.2 IPC.  Here
//   * 8 consumer warps (64 registers) each own 8 rows of the tile product and run it on the FP64
//     tensor pipe (mma.sync.m8n8k4.f64, W pre-arranged in fragment order in shared memory), decide
//     their rows in registers and load W in the shadow of the producers' first tile;
//   * 16 producer warps (88 registers) own exactly 4 chains of every 64-chain tile;
//   * the producer stages are specialised at compile time (DREAM with 3 pairs, or the
//     runtime-general form), need d % 4 == 0 so every row access is a 16-byte vector, test
//     the crossover mask on the raw Philox words against an integer threshold, and take
//     the jump statistic's 1/variance from a Newton reciprocal instead of an IEEE division.
// Draw values and proposal arithmetic are those of the other variants (identical proposals);
// the quadratic form is summed in the DMMA fragment order, so ln_like agrees with them to
// rounding (~1e-15 relative), not bit for bit.
constexpr int kV3ConsWarps = 8, kV3ProdWarps = 16;
constexpr int kV3Threads = 32 * (kV3ConsWarps + kV3ProdWarps);   // 640
constexpr int kV3ProdThreads = 32 * kV3ProdWarps;
constexpr int kV3ConsThreads = 32 * kV3ConsWarps;

__device__ __forceinline__ double2 ldg2(const double* p) { return *reinterpret_cast<const double2*>(p); }

// ---- lane -> dimension map of the write-back ----------------------------------------------
// A lane owns two 16-byte chunks of a chain row: dims {2l, 2l+1} and {64+2l, 65+2l}, so a 128-bit
// warp access covers 512 contiguous bytes = whole 32-byte sectors.  The plain map (dims 4l .. 4l+3)
// makes every access touch half of each sector, and every sector twice.  Every array the write-back
// touches is per-dimension independent, so the map is free there: 148.8 -> 141.8 us per launch
// against the plain map (profiles/r1_consumer_experiments.txt).  The proposal stage keeps the plain
// map: in the sector map the Philox words of a 4-dim slot and the jump statistic have to be passed
// between lanes by ~20 shuffles, which cost more than the halved sector count saved (153.2 against
// 143.6 us, branch exp/split-writeback).
struct WbMap {
  int o0, o1;      // element offsets of the lane's two 16-byte chunks inside a row
  bool h0, h1;     // chunk inside the row
};
__device__ __forceinline__ WbMap wb_map(int d, int lane) {
  WbMap m;
  m.o0 = 2 * lane; m.o1 = 64 + 2 * lane;
  m.h0 = m.o0 < d; m.h1 = m.o1 < d;     // d is even
  return m;
}

// NPAIR: 3 = DREAM with del_pairs == 3 (the reference default), 0 = read algo / del_pairs at run time
template <bool REPLAY, int NPAIR>
__device__ __forceinline__ void tile_stage_propose_v3(const PhaseArgs& a, const GaussTables& tb,
                                                      TileScratch& T, double* __restrict__ P, int pld,
                                                      int gwarp, int gwarps, int lane) {
  const int d = a.d;
  const bool dream = NPAIR == 3 ? true : a.algo == BPM_ALGO_DREAM;
  const int npair = NPAIR == 3 ? 3 : (dream ? a.del_pairs : 1);
  const bool act = 4 * lane < d;                      // d % 4 == 0: a lane owns 4 dims or none
  const bool adapt = dream && a.adapt;
  const bool welford_var = adapt && !(REPLAY && a.hist_base != nullptr);
  // lazy protocol (PhaseArgs::pending): the chain's CURRENT row -- already in registers here -- is the
  // history row / moment sample the previous generation left pending; it is folded in now, so the
  // kernel's tail never re-reads a moment row or a rejected chain's state
  const bool fold = a.pending && a.mean != nullptr;
  const bool need_m2 = fold || welford_var;
  for (int row = gwarp; row < kTileRows; row += gwarps) {
    const int c = T.cid[row];
    double* prow = P + row * pld + 4 * lane;          // pld even: 16-byte aligned
    if (c < 0) {
      if (act) {
        *reinterpret_cast<double2*>(prow) = make_double2(0.0, 0.0);
        *reinterpret_cast<double2*>(prow + 2) = make_double2(0.0, 0.0);
      }
      continue;
    }
    double cur[4] = {0, 0, 0, 0}, S[4] = {0, 0, 0, 0}, var[4] = {0, 0, 0, 0};
    double2 u0, u1, w0, w1, va[3][2], vb[3][2];
    if (act) {
      // every row gather of this chain is issued before anything consumes one
      const double* xc = a.X + (size_t)c * a.ld + 4 * lane;
      u0 = ldg2(xc); u1 = ldg2(xc + 2);
      if (need_m2) {
        const double* mp = a.m2 + (size_t)(c - a.chain_lo) * a.ld + 4 * lane;
        w0 = ld_stream2(mp); w1 = ld_stream2(mp + 2);        // read once per generation
      }
      if constexpr (NPAIR == 3) {
#pragma unroll
        for (int p = 0; p < 3; ++p) {
          const double* pa = a.X + (size_t)T.pa[row][p] * a.ld + 4 * lane;
          const double* pb = a.X + (size_t)T.pb[row][p] * a.ld + 4 * lane;
          va[p][0] = ldg2(pa); va[p][1] = ldg2(pa + 2);
          vb[p][0] = ldg2(pb); vb[p][1] = ldg2(pb + 2);
        }
      }
    }
    if (act) {
      if (need_m2) { var[0] = w0.x; var[1] = w0.y; var[2] = w1.x; var[3] = w1.y; }
      cur[0] = u0.x; cur[1] = u0.y; cur[2] = u1.x; cur[3] = u1.y;
      if constexpr (NPAIR == 3) {
#pragma unroll
        for (int p = 0; p < 3; ++p) {
          const double df0 = __dsub_rn(va[p][0].x, vb[p][0].x), df1 = __dsub_rn(va[p][0].y, vb[p][0].y);
          const double df2 = __dsub_rn(va[p][1].x, vb[p][1].x), df3 = __dsub_rn(va[p][1].y, vb[p][1].y);
          S[0] = p == 0 ? df0 : __dadd_rn(S[0], df0);
          S[1] = p == 0 ? df1 : __dadd_rn(S[1], df1);
          S[2] = p == 0 ? df2 : __dadd_rn(S[2], df2);
          S[3] = p == 0 ? df3 : __dadd_rn(S[3], df3);
        }
      } else {
        for (int p = 0; p < npair; ++p) {
          const double* pa = a.X + (size_t)T.pa[row][p] * a.ld + 4 * lane;
          const double* pb = a.X + (size_t)T.pb[row][p] * a.ld + 4 * lane;
          const double2 s0 = ldg2(pa), s1 = ldg2(pa + 2), t0 = ldg2(pb), t1 = ldg2(pb + 2);
          const double df0 = __dsub_rn(s0.x, t0.x), df1 = __dsub_rn(s0.y, t0.y);
          const double df2 = __dsub_rn(s1.x, t1.x), df3 = __dsub_rn(s1.y, t1.y);
          S[0] = p == 0 ? df0 : __dadd_rn(S[0], df0);
          S[1] = p == 0 ? df1 : __dadd_rn(S[1], df1);
          S[2] = p == 0 ? df2 : __dadd_rn(S[2], df2);
          S[3] = p == 0 ? df3 : __dadd_rn(S[3], df3);
        }
      }
    }
    // the partner rows are consumed: their landing registers now take the mean row, whose latency hides
    // behind the draws below; the pending history row leaves straight from the registers
    double2 mn0 = make_double2(0.0, 0.0), mn1 = mn0;
    if (act && a.pending) {
      const size_t o = (size_t)(c - a.chain_lo) * a.ld + 4 * lane;
      if (fold) { mn0 = ld_stream2(a.mean + o); mn1 = ld_stream2(a.mean + o + 2); }
      if (a.hist_cur) {
        st_stream2(a.hist_cur + o, cur[0], cur[1]);
        st_stream2(a.hist_cur + o + 2, cur[2], cur[3]);
      }
    }
    uint32_t mbits = 0xFu;
    double gamma;
    const double gu = T.gamma_u[row];
    if (dream) {
      mbits = 0u;
      const int m = T.cr_idx[row];
      if (act) {
        if (REPLAY) {
          const double cr = tb.crv[m];
          double z[4];
          z4<REPLAY>(a, c, lane, z);
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (z[q] <= cr) mbits |= 1u << q;
        } else {
          const uint32_t th = tb.thr[m];
          mbits = zen_mask4(draw4(a.rng, (uint32_t)c, RNG_ZEN, (uint32_t)lane), th);
        }
      }
      int d_prime = __reduce_add_sync(0xFFFFFFFFu, __popc(mbits));
      if (d_prime == 0) {
        const int fb = T.fallback[row] < 0 ? 0 : T.fallback[row];
        if ((fb >> 2) == lane) mbits |= 1u << (fb & 3);
        d_prime = 1;
      }
      gamma = tb.gam[d_prime];
      if (a.gamma_jump) gamma = gu < a.gamma_p0 ? gamma : 1.0;
    } else {
      gamma = demc_gamma(a, gu);
    }
    double delta = 0.0;
    if (act) {
      double e[4], nn[4], prv[4];
      en4<REPLAY>(a, c, lane, e, nn);
      if (fold) {
        // Welford update with the pending row (same arithmetic, same order as an eager write-back):
        // afterwards var[] / mom_len is np.std(chain.chain)^2 over the whole history (dream.py:128)
        welford_update(cur[0], a.inv_mom, mn0.x, var[0]);
        welford_update(cur[1], a.inv_mom, mn0.y, var[1]);
        welford_update(cur[2], a.inv_mom, mn1.x, var[2]);
        welford_update(cur[3], a.inv_mom, mn1.y, var[3]);
        const size_t o = (size_t)(c - a.chain_lo) * a.ld + 4 * lane;
        st_stream2(a.mean + o, mn0.x, mn0.y); st_stream2(a.mean + o + 2, mn1.x, mn1.y);
        st_stream2(a.m2 + o, var[0], var[1]); st_stream2(a.m2 + o + 2, var[2], var[3]);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        double pr;
        if (dream) {
          pr = dream_prop(cur[q], S[q], e[q], nn[q], gamma, (mbits >> q) & 1u ? 1.0 : 0.0);
          if (adapt) {
            double v;
            if (welford_var) {
              v = __dmul_rn(var[q], a.inv_mom);
              if (!(v > 0.0)) v = 1e-12 * 1e-12;
            } else {
              v = cr_variance<REPLAY>(a, c, 4 * lane + q);
            }
            delta += cr_term(cur[q], pr, v);
          }
        } else {
          pr = demc_prop(cur[q], S[q], nn[q], gamma);
        }
        prv[q] = pr;
      }
      *reinterpret_cast<double2*>(prow) = make_double2(prv[0], prv[1]);
      *reinterpret_cast<double2*>(prow + 2) = make_double2(prv[2], prv[3]);
      if (REPLAY && a.tr.prop) {          // replay trace: the proposal vector the reference built (dream.py:85-89)
        double* tp = a.tr.prop + (size_t)c * d + 4 * lane;
#pragma unroll
        for (int q = 0; q < 4; ++q) tp[q] = prv[q];
      }
    }
    if (dream) {
      delta = group_sum_d<32>(delta);
      if (lane == 0) {
        a.cr_pick[c] = adapt ? T.cr_idx[row] : -1;
        a.cr_delta[c] = delta;
      }
    }
  }
}

// ---- mbarrier helpers (CTA scope): variant 3 hands tiles over with these so that no producer
// warp ever waits for another producer warp -------------------------------------------------
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* b, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
  asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_addr(b)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.acquire.cta.shared::cta.b64 p, [%1], %2, 0x1000;\n"
                 "selp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(smem_addr(b)), "r"(parity) : "memory");
  }
}

// Per-warp scalar draws: producer warp pw owns tile rows pw, pw + 16, pw + 32, pw + 48 from the
// draws to the write-back, so the scratch of a row is written and read by one warp only (plus
// the consumers, ordered by the FULL mbarrier).  gid0 = population-list index of tile row 0,
// gid_end = end of this CTA's row range.  No L2 prefetch of the rows a tile will touch: with 16
// independent producer warps it no longer pays -- the kernel is 9 % faster without it
// (profiles/r1_ab_prefetch.txt).
template <bool REPLAY>
__device__ __forceinline__ void warp_stage_draws(const PhaseArgs& a, const PhaseLists& L,
                                                 const GaussTables& tb, TileScratch& T, int gid0,
                                                 int gid_end, int pw, int lane) {
  const bool dream = a.algo == BPM_ALGO_DREAM;
  const int npair = dream ? a.del_pairs : 1;
  const int nslots = 2 + npair;
  const int rows_per_warp = kTileRows / kV3ProdWarps;
  for (int idx = lane; idx < rows_per_warp * nslots; idx += 32) {
    const int j = idx / nslots, slot = idx - j * nslots;
    const int row = pw + kV3ProdWarps * j;
    const int gid = gid0 + row;
    bool valid = gid < gid_end;
    const int c = valid ? L.self[gid] : 0;
    valid = valid && c >= a.chain_lo && c < a.chain_hi;
    if (slot == 0) T.cid[row] = valid ? c : -1;
    if (!valid) continue;
    if (REPLAY) {
      if (slot == 0) {
        T.cr_idx[row] = dream ? a.rp.cr_idx[c] : 0;
        T.accept_u[row] = a.rp.accept_u[c];
      } else if (slot == 1) {
        T.gamma_u[row] = a.rp.gamma_u[c];
        T.fallback[row] = dream ? a.rp.fallback_dim[c] : -1;
      } else {
        const int p = slot - 2;
        T.pa[row][p] = L.pool[a.rp.pairs[((size_t)c * npair + p) * 2 + 0]];
        T.pb[row][p] = L.pool[a.rp.pairs[((size_t)c * npair + p) * 2 + 1]];
      }
    } else {
      const Philox4 q = draw4(a.rng, (uint32_t)c, RNG_SCALAR, (uint32_t)slot);
      if (slot == 0) {
        int m = 0;
        if (dream) {
          const double u = slot0_cr_u(q);
          for (int jj = 0; jj < a.n_cr; ++jj)
            if (tb.cdf[jj] <= u) m = jj + 1;
          m = m < a.n_cr ? m : a.n_cr - 1;
        }
        T.cr_idx[row] = m;
        T.accept_u[row] = slot0_accept_u(q);
      } else if (slot == 1) {
        T.gamma_u[row] = slot1_gamma_u(q);
        T.fallback[row] = slot1_fallback(q, a.d);
      } else {
        int r1, r2;
        slot_pair(q, L.n_pool, r1, r2);
        BPM_CHECK(r1 >= 0 && r1 < L.n_pool && r2 >= 0 && r2 < L.n_pool && r1 != r2, "pair draw", r1 * 100000LL + r2);
        const int ga = L.pool[r1], gb = L.pool[r2];
        BPM_CHECK(ga >= 0 && ga < a.N && gb >= 0 && gb < a.N, "partner chain id", ga);
        T.pa[row][slot - 2] = ga;
        T.pb[row][slot - 2] = gb;
      }
    }
  }
  __syncwarp();
}

// Accepted rows leave the tile from the CONSUMER warp that decided them: the proposal row is still in
// shared memory, the stores need no landing registers and nobody waits for them.  Lane map = wb_map
// (whole 32-byte sectors per warp access).  Rejected chains cost nothing here: their state, history row
// and moments are handled by the lazy protocol in the next generation's proposal stage.
__device__ __forceinline__ void cons_store_row(const PhaseArgs& a, const double* __restrict__ prow, int c,
                                               const WbMap& mp) {
  const size_t ox = (size_t)c * a.ld;
  if (mp.h0) {
    const double2 x = *reinterpret_cast<const double2*>(prow + mp.o0);
    *reinterpret_cast<double2*>(a.X + ox + mp.o0) = x;
    store_peers2(a, ox + mp.o0, x.x, x.y);
  }
  if (mp.h1) {
    const double2 x = *reinterpret_cast<const double2*>(prow + mp.o1);
    *reinterpret_cast<double2*>(a.X + ox + mp.o1) = x;
    store_peers2(a, ox + mp.o1, x.x, x.y);
  }
}

__host__ __device__ inline size_t v3_ptile_doubles(int d) { return (size_t)kTileRows * dmma_pld(d) + kTileRows; }
inline size_t fused_v3_smem(int d) {
  return sizeof(double) * (gauss_table_doubles(d) + 2 * v3_ptile_doubles(d) + 3 * gauss_scratch_doubles() + 4);
}
template <bool REPLAY, bool CENTER, int NPAIR>
__global__ void __launch_bounds__(kV3Threads, 1)
fused_gauss_v3_kernel(const PhaseArgs a, const GaussArgs g) {
  extern __shared__ __align__(16) double smem[];
  const int d = a.d, pld = dmma_pld(d), NT = dmma_ntiles(g.r);
  const GaussTables tb = carve_tables(smem, d);      // tb.Ws holds W in DMMA fragment order
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* Pbuf = smem + gauss_table_doubles(d);
  const size_t p_stride = v3_ptile_doubles(d);
  double* Tbuf = Pbuf + 2 * p_stride;
  const size_t t_stride = gauss_scratch_doubles();
  uint64_t* bars = reinterpret_cast<uint64_t*>(Tbuf + 3 * t_stride);
  uint64_t* FULL = bars;       // [2] every producer warp filled its rows of the tile buffer
  uint64_t* DONE = bars + 2;   // [2] every row of the tile is decided (T.acc, lnl final)
  fill_tables_v3(a, g, tb, threadIdx.x, kV3Threads);
  if (threadIdx.x == 0) {
    mbar_init(FULL + 0, kV3ProdWarps); mbar_init(FULL + 1, kV3ProdWarps);   // one arrival per producer warp
    mbar_init(DONE + 0, kTileRows); mbar_init(DONE + 1, kTileRows);         // one per deciding thread
  }
  __syncthreads();
  const PhaseLists L = phase_lists(a);
  // every CTA owns an equal contiguous range of the phase list (no 5-vs-6-tile imbalance):
  // full 64-row tiles plus one partial tile
  const int per_cta = (L.n_self + (int)gridDim.x - 1) / (int)gridDim.x;
  const int g_lo = min((int)blockIdx.x * per_cta, L.n_self);
  const int g_hi = min(g_lo + per_cta, L.n_self);
  const int n_my = (g_hi - g_lo + kTileRows - 1) / kTileRows;

  if (warp < kV3ConsWarps) {
    // ------------------------------ consumers ------------------------------------------
    // 8 warps x 8 rows: tile product on the FP64 tensor pipe, Metropolis decision and DONE arrival
    // all inside the warp.  768 threads launch with 80 registers each; the consumers hand 16 of
    // theirs to the producers (16 x 88 + 8 x 64 = 24 x 80: setmaxnreg only moves registers inside
    // the CTA's allocation).  They also load W, in the shadow of the producers' first tile.
    asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
    load_W_fragments(tb.Ws, tb.mus, g.W, g.mu, d, g.r, threadIdx.x, kV3ConsThreads);
    nbar_sync(BAR_CONS, kV3ConsThreads);
    unsigned n_acc = 0, n_rej = 0;
    const WbMap mp = wb_map(d, lane);
    for (int i = 0; i < n_my; ++i) {
      const int b = i & 1;
      const double* P = Pbuf + b * p_stride;
      TileScratch& T = *reinterpret_cast<TileScratch*>(Tbuf + (i % 3) * t_stride);
      mbar_wait(FULL + b, (i >> 1) & 1);
      const double maha = gauss_tile_maha_dmma8<CENTER>(P, pld, tb.Ws, tb.mus, d, NT, warp, lane);
      const bool decider = (lane & 3) == 0;
      const int acc = tile_stage_decide_reg(a, g, T, maha, decider ? 8 * warp + (lane >> 2) : -1, n_acc, n_rej);
      unsigned am = __ballot_sync(0xFFFFFFFFu, decider && acc);
      while (am) {                                   // ~1 accepted row per 8-row m-tile
        const int row = 8 * warp + ((__ffs(am) - 1) >> 2);
        am &= am - 1;
        cons_store_row(a, P + row * pld, T.cid[row], mp);
      }
      __syncwarp();                                  // the tile reads above precede the buffer's release
      if (decider) mbar_arrive(DONE + b);
    }
    if (lane == 0) {
      if (n_acc) atomicAdd(a.n_acc, (unsigned long long)n_acc);
      if (n_rej) atomicAdd(a.n_rej, (unsigned long long)n_rej);
    }
  } else {
    // ------------------------------ producers ------------------------------------------
    // each warp is an independent pipeline over ITS rows: draws of tile i+1 | proposal of tile i; it
    // synchronises only with the consumers (FULL: tile handed over; DONE: tile buffer and scratch slot of
    // tile i-2 are free again -- the consumers decided it and stored its accepted rows)
    asm volatile("setmaxnreg.inc.sync.aligned.u32 88;");
    const int pw = warp - kV3ConsWarps;
    if (n_my > 0)
      warp_stage_draws<REPLAY>(a, L, tb, *reinterpret_cast<TileScratch*>(Tbuf), g_lo, g_hi, pw, lane);
    for (int i = 0; i < n_my; ++i) {
      const int b = i & 1;
      // scratch slot (i + 1) % 3 was tile i-2's
      if (i >= 2) mbar_wait(DONE + b, ((i - 2) >> 1) & 1);
      if (i + 1 < n_my)
        warp_stage_draws<REPLAY>(a, L, tb, *reinterpret_cast<TileScratch*>(Tbuf + ((i + 1) % 3) * t_stride),
                                 g_lo + (i + 1) * kTileRows, g_hi, pw, lane);
      double* P = Pbuf + b * p_stride;
      TileScratch& T = *reinterpret_cast<TileScratch*>(Tbuf + (i % 3) * t_stride);
      tile_stage_propose_v3<REPLAY, NPAIR>(a, tb, T, P, pld, pw, kV3ProdWarps, lane);
      __syncwarp();
      if (lane == 0) mbar_arrive(FULL + b);
    }
  }
}

template <bool REPLAY, bool CENTER, int NPAIR>
inline int launch_fused_v3(const PhaseArgs& a, const GaussArgs& g, int grid, size_t sm, cudaStream_t s) {
  cudaError_t e = cudaFuncSetAttribute(fused_gauss_v3_kernel<REPLAY, CENTER, NPAIR>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
  if (e != cudaSuccess) return 1;
  fused_gauss_v3_kernel<REPLAY, CENTER, NPAIR><<<grid, kV3Threads, sm, s>>>(a, g);
  return 0;
}

}  // namespace bpm
#include "kernels_fused_v4.cuh"     // fused_gauss_v4_kernel: v3 with TMA-staged partner gathers (uses the helpers above)
namespace bpm {

// The fused Gaussian half-phase kernel of a configuration, decided here and nowhere else: the engine plans the
// lazy protocol from it before it builds the phase arguments (v3 and v4 leave the generation's new history row /
// moment sample pending, PhaseArgs::lazy; ws writes them eagerly), and try_fused_phase launches it.  Shared memory
// (227 KB per CTA) decides which kernels exist for a d: d = 108 fits v3 only, d = 112 none.
//   1. none, unless the target is the Gaussian, gauss_rows_supported(d, r) holds and ld is even;
//   2. ws, if fused_gauss_smem(d) fits and either mode is BPM_FUSED_GAUSS_WS or the v3 conditions below fail;
//   3. if the v3 conditions hold (d % 4 == 0, ld == d, fused_v3_smem(d) fits): v4 when mode is not
//      BPM_FUSED_GAUSS_V3 and fused_v4_fits(d, ld, r, npair) holds, otherwise v3;
//   4. none otherwise (d = 112): the engine runs the split path.
// npair: del_pairs for DREAM, 1 for DE-MC.  mode: bpm_set_fused's value (not BPM_FUSED_OFF).
enum class GaussKernel { none, ws, v3, v4 };
inline GaussKernel gauss_fused_kernel(int target, int d, int ld, int r, int npair, int mode) {
  if (!(target == BPM_TARGET_GAUSS && gauss_rows_supported(d, r) && (ld % 2) == 0)) return GaussKernel::none;
  const bool v3_ok = (d % 4) == 0 && ld == d && fused_v3_smem(d) <= kMaxDynSmem;
  if (fused_gauss_smem(d) <= kMaxDynSmem && (mode == BPM_FUSED_GAUSS_WS || !v3_ok)) return GaussKernel::ws;
  if (v3_ok)
    return mode != BPM_FUSED_GAUSS_V3 && fused_v4_fits(d, ld, r, npair) ? GaussKernel::v4 : GaussKernel::v3;
  return GaussKernel::none;
}

// One fused half-phase: the Gaussian kernel gk names (gauss_fused_kernel), or fused_small_kernel for the d <= 4
// analytic targets.  *done = 0: nothing was launched, the caller runs the split path.
template <bool REPLAY>
inline int try_fused_phase(const TargetView& tv, const PhaseArgs& a, cudaStream_t s, GaussKernel gk, int* done) {
  *done = 0;
  if (gk != GaussKernel::none) {
    GaussArgs g;
    g.mu = tv.mu; g.W = tv.W; g.Wf = tv.Wf; g.r = tv.r; g.c0 = tv.c0; g.log_of_pdf = tv.log_of_pdf;
    const int n_tiles = (a.nA + kTileRows - 1) / kTileRows;
    const int grid = n_tiles > 148 ? 148 : (n_tiles < 1 ? 1 : n_tiles);
    if (gk == GaussKernel::ws) {
      const size_t sm = fused_gauss_smem(a.d);
      cudaError_t e;
      if (tv.mu_is_zero) {
        e = cudaFuncSetAttribute(fused_gauss_ws_kernel<REPLAY, false>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        if (e != cudaSuccess) return 1;
        fused_gauss_ws_kernel<REPLAY, false><<<grid, kWsThreads, sm, s>>>(a, g);
      } else {
        e = cudaFuncSetAttribute(fused_gauss_ws_kernel<REPLAY, true>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        if (e != cudaSuccess) return 1;
        fused_gauss_ws_kernel<REPLAY, true><<<grid, kWsThreads, sm, s>>>(a, g);
      }
    } else {
      const bool d3 = a.algo == BPM_ALGO_DREAM && a.del_pairs == 3;
      int rc;
      if (gk == GaussKernel::v4) {        // TMA-staged gathers
        const int npair = a.algo == BPM_ALGO_DREAM ? a.del_pairs : 1;
        const size_t sm4 = v4_layout(a.d, tv.r, npair).total;
        const bool d1 = a.algo == BPM_ALGO_DEMC;
        if (tv.mu_is_zero)
          rc = d3 ? launch_fused_v4<REPLAY, false, 3>(a, g, grid, sm4, s)
             : d1 ? launch_fused_v4<REPLAY, false, 1>(a, g, grid, sm4, s)
                  : launch_fused_v4<REPLAY, false, 0>(a, g, grid, sm4, s);
        else
          rc = d3 ? launch_fused_v4<REPLAY, true, 3>(a, g, grid, sm4, s)
             : d1 ? launch_fused_v4<REPLAY, true, 1>(a, g, grid, sm4, s)
                  : launch_fused_v4<REPLAY, true, 0>(a, g, grid, sm4, s);
      } else {                            // v3: register gathers
        const size_t sm = fused_v3_smem(a.d);
        if (tv.mu_is_zero)
          rc = d3 ? launch_fused_v3<REPLAY, false, 3>(a, g, grid, sm, s)
                  : launch_fused_v3<REPLAY, false, 0>(a, g, grid, sm, s);
        else
          rc = d3 ? launch_fused_v3<REPLAY, true, 3>(a, g, grid, sm, s)
                  : launch_fused_v3<REPLAY, true, 0>(a, g, grid, sm, s);
      }
      if (rc) return 1;
    }
    if (cudaGetLastError() != cudaSuccess) return 1;
    *done = 1;
    return 0;
  }
  if (a.d <= 4 && (tv.target == BPM_TARGET_BANANA || tv.target == BPM_TARGET_BIMODAL ||
                   tv.target == BPM_TARGET_LINEFIT)) {
    const int grid = (a.nA + 127) / 128;
    // (Programmatic dependent launches between phase a, phase b and the CR reduction -- griddepcontrol.wait after
    // the list lookups, launch_dependents at the top -- were measured and dropped: 10^5 line-fit chains 52.6 -> 59.7 us
    // per generation, 10^6 bimodal chains 241 -> 264 us; profiles/r2/r2z_secondary*.txt.)
    if (tv.target == BPM_TARGET_BANANA)
      fused_small_kernel<REPLAY, BPM_TARGET_BANANA><<<grid, 128, 0, s>>>(a, tv);
    else if (tv.target == BPM_TARGET_BIMODAL)
      fused_small_kernel<REPLAY, BPM_TARGET_BIMODAL><<<grid, 128, 0, s>>>(a, tv);
    else
      fused_small_kernel<REPLAY, BPM_TARGET_LINEFIT>
          <<<grid, 128, sizeof(double) * 3 * tv.linefit_M, s>>>(a, tv);
    if (cudaGetLastError() != cudaSuccess) return 1;
    *done = 1;
    return 0;
  }
  return 0;
}

}  // namespace bpm
