// Generic (any d, any likelihood) split path of one half-phase:
//   propose_kernel  -> prop[n_self][ld]           (demc.py:161-182 / dream.py:40-93)
//   <likelihood>    -> lnl_prop[n_self]            (samplers.py:330)
//   accept_kernel   -> X, lnl, moments, history    (samplers.py:328-336, demc.py:188-196)
// A group of LPC lanes (1, 4, 8 or 32) owns one chain; each lane owns dimension blocks
// of four consecutive doubles, b = sub + t * LPC.  The fused single-kernel variants in
// kernels_fused.cuh reuse the same draw / arithmetic helpers (step.cuh), so both paths
// produce bit-identical chains.
#pragma once
#include "step.cuh"
#include "targets.cuh"

namespace bpm {

constexpr int kMaxBlocksPerLane = 8;  // d <= 4 * 8 * LPC  (1024 at LPC = 32)
constexpr int kThreads = 256;

// ---- demc.py:81-100: flip coin + shuffled split (native RNG) ----------------------
__global__ void split_native_kernel(int32_t* __restrict__ perm, int32_t* __restrict__ inv,
                                    int32_t* __restrict__ flip, int N, int shuffle, double flip_p, RngCtx rng,
                                    int inv_lo, int inv_hi) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j == 0) {
    Philox4 q = draw4(rng, 0xFFFFFFFFu, RNG_GEN, 0);
    double thr = __ddiv_rn(flip_p, __dadd_rn(flip_p, __dsub_rn(1.0, flip_p)));
    *flip = u53(q.x, q.y) < thr ? 1 : 0;
  }
  // the Feistel keys cost two Philox calls: drawn once per block, not once per element
  __shared__ FeistelKey fkey;
  if (shuffle && threadIdx.x == 0) fkey = make_feistel(rng, (uint32_t)N);
  __syncthreads();
  if (j >= N) return;
  int32_t c = j;
  if (shuffle) c = (int32_t)feistel_perm(fkey, (uint32_t)j);
  perm[j] = c;
  if (inv && c >= inv_lo && c < inv_hi) inv[c] = j;   // list position of chain c (packs the phase lists in chain order)
}
__global__ void invert_perm_kernel(const int32_t* __restrict__ perm, int32_t* __restrict__ inv, int N) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < N) inv[perm[j]] = j;
}

__global__ void set_flag_kernel(int32_t* flag, int32_t v) { *flag = v; }
__global__ void identity_split_kernel(int32_t* __restrict__ perm, int32_t* __restrict__ inv,
                                      int32_t* __restrict__ flip, int N) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j == 0) *flip = 0;
  if (j < N) {
    perm[j] = j;
    if (inv) inv[j] = j;
  }
}

// number of rows of the half being stepped, picked on the device (the flip flag lives there)
__global__ void phase_count_kernel(const int32_t* __restrict__ loc_cnt, const int32_t* __restrict__ flip, int phase,
                                   int serial, int32_t* __restrict__ out) {
  const int first = serial ? 1 : ((phase ^ (*flip != 0)) == 0);
  *out = loc_cnt[first ? 0 : 1];
}

// ---- packed phase lists: the chains this rank owns, per half, in CHAIN order ----------
// A rank steps only its own chains (demc.py:103-107 loops over the local ids and tests
// `c_id in a_ids`).  Walking the global half-lists and skipping foreign chains would leave
// every 64-chain tile 1/G full on G GPUs, so each generation the local members of the two
// halves are packed into loc_list with three small kernels (per-block counts, a one-block
// scan, per-block write) that walk the LOCAL chains c in [lo, hi) in ascending order and
// look their half up in the inverse permutation.  Chain order also makes every per-chain
// access of a phase kernel (own row, moments, cached lnL, CR slots) monotone in memory, which
// is what the 16-byte rows of the d <= 4 targets need to share 32-byte sectors; unsharded
// small-d handles use the packed lists for that reason alone.
constexpr int kCompactThreads = 256, kCompactPer = 8, kCompactBlock = kCompactThreads * kCompactPer;
// exclusive prefix sums of (xa, xb) over the threads of a block (NT <= 1024), warp shuffles + one smem hop
template <int NT>
__device__ __forceinline__ void block_excl_scan2(int xa, int xb, int& ea, int& eb, int& tota, int& totb) {
  __shared__ int wa[NT / 32], wb[NT / 32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int ia = xa, ib = xb;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int ya = __shfl_up_sync(0xFFFFFFFFu, ia, o), yb = __shfl_up_sync(0xFFFFFFFFu, ib, o);
    if (lane >= o) { ia += ya; ib += yb; }
  }
  if (lane == 31) { wa[w] = ia; wb[w] = ib; }
  __syncthreads();
  if (w == 0) {
    int va = lane < NT / 32 ? wa[lane] : 0, vb = lane < NT / 32 ? wb[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int ya = __shfl_up_sync(0xFFFFFFFFu, va, o), yb = __shfl_up_sync(0xFFFFFFFFu, vb, o);
      if (lane >= o) { va += ya; vb += yb; }
    }
    if (lane < NT / 32) { wa[lane] = va; wb[lane] = vb; }     // inclusive over warps
  }
  __syncthreads();
  ea = ia - xa + (w > 0 ? wa[w - 1] : 0);
  eb = ib - xb + (w > 0 ? wb[w - 1] : 0);
  tota = wa[NT / 32 - 1];
  totb = wb[NT / 32 - 1];
}
// inv[c]: where chain c sits in the shuffled list
__device__ __forceinline__ void compact_flags(const int32_t* inv, int nA, int hi, int c0, int& cA,
                                              int& cB, unsigned& mA, unsigned& mB) {
  cA = cB = 0; mA = mB = 0u;
#pragma unroll
  for (int k = 0; k < kCompactPer; ++k) {
    const int c = c0 + k;
    if (c < hi) {
      if (inv[c] < nA) { ++cA; mA |= 1u << k; } else { ++cB; mB |= 1u << k; }
    }
  }
}
__global__ void __launch_bounds__(kCompactThreads) compact_count_kernel(const int32_t* inv,
                                                                        int nA, int lo, int hi,
                                                                        int32_t* __restrict__ blk_cnt) {
  __shared__ int sa[kCompactThreads / 32], sb[kCompactThreads / 32];
  int cA, cB; unsigned mA, mB;
  compact_flags(inv, nA, hi, lo + blockIdx.x * kCompactBlock + threadIdx.x * kCompactPer, cA, cB, mA, mB);
  cA = __reduce_add_sync(0xFFFFFFFFu, cA);
  cB = __reduce_add_sync(0xFFFFFFFFu, cB);
  if ((threadIdx.x & 31) == 0) { sa[threadIdx.x >> 5] = cA; sb[threadIdx.x >> 5] = cB; }
  __syncthreads();
  if (threadIdx.x == 0) {
    int ta = 0, tb = 0;
    for (int w = 0; w < kCompactThreads / 32; ++w) { ta += sa[w]; tb += sb[w]; }
    blk_cnt[2 * blockIdx.x] = ta;
    blk_cnt[2 * blockIdx.x + 1] = tb;
  }
}
// exclusive scan of the block counts (one block; thread t owns a contiguous run of blocks)
__global__ void __launch_bounds__(1024) compact_scan_kernel(const int32_t* __restrict__ blk_cnt, int nblk,
                                                            int32_t* __restrict__ blk_off,
                                                            int32_t* __restrict__ tot) {
  const int per = (nblk + 1023) / 1024;
  const int b0 = threadIdx.x * per, b1 = min(nblk, b0 + per);
  int ta = 0, tb = 0;
  for (int b = b0; b < b1; ++b) { ta += blk_cnt[2 * b]; tb += blk_cnt[2 * b + 1]; }
  int ra, rb, alla, allb;
  block_excl_scan2<1024>(ta, tb, ra, rb, alla, allb);
  if (threadIdx.x == 0) { tot[0] = alla; tot[1] = allb; }
  for (int b = b0; b < b1; ++b) {
    blk_off[2 * b] = ra; blk_off[2 * b + 1] = rb;
    ra += blk_cnt[2 * b]; rb += blk_cnt[2 * b + 1];
  }
}
__global__ void __launch_bounds__(kCompactThreads) compact_write_kernel(const int32_t* inv,
                                                                        int nA, int lo, int hi,
                                                                        const int32_t* __restrict__ blk_off,
                                                                        int32_t* __restrict__ loc_list) {
  const int c0 = lo + blockIdx.x * kCompactBlock + threadIdx.x * kCompactPer;
  int cA, cB; unsigned mA, mB;
  compact_flags(inv, nA, hi, c0, cA, cB, mA, mB);
  int ea, eb, ta, tb;
  block_excl_scan2<kCompactThreads>(cA, cB, ea, eb, ta, tb);
  int oa = blk_off[2 * blockIdx.x] + ea;
  int ob = nA + blk_off[2 * blockIdx.x + 1] + eb;
#pragma unroll
  for (int k = 0; k < kCompactPer; ++k) {
    if (mA & (1u << k)) loc_list[oa++] = c0 + k;
    if (mB & (1u << k)) loc_list[ob++] = c0 + k;
  }
}

// ---- proposal ---------------------------------------------------------------------
// PROB (multi-problem handles, pb used): the chain of slot gid comes from problem_slot, and its draws are
// addressed by the problem's key, the chain's index within the problem and the problem's p_cr row.
__device__ __forceinline__ PhaseLists slot_lists(const ProblemSlot& ps) {
  PhaseLists L;
  L.self = nullptr; L.n_self = 0; L.skip_self = 0;
  L.pool = ps.pool; L.n_pool = ps.n_pool;
  return L;
}
template <bool REPLAY, int LPC, bool PROB = false>
// (LPC = 32: two 256-thread blocks per SM, i.e. at most 128 registers -- without the bound the block-wise pass 2
// takes 174 and one block per SM)
__global__ void __launch_bounds__(kThreads, LPC == 32 ? 2 : 1) propose_kernel(const PhaseArgs a, const ProblemArgs prob) {
  const int gid = (blockIdx.x * kThreads + threadIdx.x) / LPC;
  const int sub = threadIdx.x % LPC;
  ProblemSlot ps;
  if constexpr (PROB) ps = problem_slot(a, prob, gid);
  const PhaseLists L = PROB ? slot_lists(ps) : phase_lists(a);
  bool valid = PROB ? ps.valid : gid < L.n_self;
  const int c = PROB ? ps.c : (valid ? L.self[gid] : 0);
  if constexpr (!PROB) valid = valid && c >= a.chain_lo && c < a.chain_hi;
  const bool dream = a.algo == BPM_ALGO_DREAM;
  const int nblk = (a.d + 3) >> 2;

  ChainDraws D;
  D.cr_idx = 0; D.fallback = -1; D.gamma_u = 0.0;
  if (valid) {
    if constexpr (PROB) chain_scalar_draws<REPLAY>(a, ps.rng, ps.p_cr, c, ps.j, L.n_pool, D);
    else chain_scalar_draws<REPLAY>(a, c, L.n_pool, D);
  }

  // pass 1 (DREAM): crossover mask of this lane's dimensions, d' (dream.py:51-58)
  uint32_t mbits = 0xFFFFFFFFu;
  double gamma;
  // large d (one warp per chain, rows of whole 32-byte sectors): pass 2 below works block-wise with 16-byte
  // accesses and reuses pass 1's Philox words
  constexpr bool kKeepDraws = LPC == 32 && !REPLAY;
  const bool vec = LPC == 32 && (a.ld & 3) == 0;
  Philox4 qs[kKeepDraws ? kMaxBlocksPerLane : 1];
  if (dream) {
    mbits = 0u;
    const double cr = __ddiv_rn((double)(D.cr_idx + 1), (double)a.n_cr);
    if (valid) {
#pragma unroll
      for (int t = 0; t < kMaxBlocksPerLane; ++t) {
        const int b = sub + t * LPC;
        if (b < nblk) {
          double z[4];
          if constexpr (kKeepDraws) {          // z4's native branch, keeping the call's words for zen_en4
            const Philox4 q = PROB ? draw4(ps.rng, (uint32_t)ps.j, RNG_ZEN, (uint32_t)b)
                                   : draw4(a.rng, (uint32_t)c, RNG_ZEN, (uint32_t)b);
            qs[t] = q;
            zen_z4(q, z);
          } else {
            if constexpr (PROB) z4<REPLAY>(a, ps.rng, c, ps.j, b, z);
            else z4<REPLAY>(a, c, b, z);
          }
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (4 * b + q < a.d && z[q] <= cr) mbits |= 1u << (4 * t + q);
        }
      }
    }
    int d_prime = group_sum_i<LPC>(__popc(mbits));
    if (d_prime == 0) {  // dream.py:55-57: one random dimension
      const int fdim = D.fallback < 0 ? 0 : D.fallback;
      const int fb = fdim >> 2;
      if (valid && (fb % LPC) == sub) mbits |= 1u << (4 * (fb / LPC) + (fdim & 3));
      d_prime = 1;
    }
    gamma = dream_gamma(a, d_prime, D.gamma_u);
  } else {
    gamma = demc_gamma(a, D.gamma_u);
  }

  // pass 2: gather partner rows, build the proposal
  const int npair = dream ? a.del_pairs : 1;
  const double* pa[BPM_MAX_PAIRS];
  const double* pb[BPM_MAX_PAIRS];
#pragma unroll
  for (int p = 0; p < BPM_MAX_PAIRS; ++p) {
    pa[p] = a.X; pb[p] = a.X;
    if (valid && p < npair) {
      pa[p] = a.X + (size_t)pool_chain(L, D.r1[p], c) * a.ld;
      pb[p] = a.X + (size_t)pool_chain(L, D.r2[p], c) * a.ld;
    }
  }
  const double* xc = a.X + (size_t)c * a.ld;
  double* out = a.prop + (size_t)gid * a.ld;
  double delta = 0.0;
  if (valid && vec) {
    // Block-wise: ALL loads of a 4-dim block (own row, 2 * npair partner rows, the M2 row) are issued as 16-byte
    // loads before anything of the block is stored.  The per-dimension form below stores out[i] before it loads
    // dimension i + 1 -- the pointers may alias as far as the compiler knows -- so every load's latency was
    // exposed: d = 1000, 10^4 chains per launch: 234 us, DRAM at 19 % (profiles/r2/r2x_c5_propose_accept_ncu.txt).
    // Same arithmetic per dimension, same order of the per-lane sum `delta`.
    const bool hist_var = REPLAY && a.hist_base != nullptr;
    const bool adapt = dream && a.adapt;
    const double* m2row = a.m2 + (size_t)(c - a.chain_lo) * a.ld;     // read only when adapt && !hist_var
#pragma unroll
    for (int t = 0; t < kMaxBlocksPerLane; ++t) {
      const int b = sub + t * LPC;
      if (b < nblk) {
        const int i0 = 4 * b;
        const double2 c0 = *reinterpret_cast<const double2*>(xc + i0);
        const double2 c1 = *reinterpret_cast<const double2*>(xc + i0 + 2);
        double2 w0 = make_double2(0.0, 0.0), w1 = w0;
        if (adapt && !hist_var) {
          w0 = *reinterpret_cast<const double2*>(m2row + i0);
          w1 = *reinterpret_cast<const double2*>(m2row + i0 + 2);
        }
        double S[4];
        {
          const double2 s0 = *reinterpret_cast<const double2*>(pa[0] + i0);
          const double2 s1 = *reinterpret_cast<const double2*>(pa[0] + i0 + 2);
          const double2 t0 = *reinterpret_cast<const double2*>(pb[0] + i0);
          const double2 t1 = *reinterpret_cast<const double2*>(pb[0] + i0 + 2);
          S[0] = __dsub_rn(s0.x, t0.x); S[1] = __dsub_rn(s0.y, t0.y);
          S[2] = __dsub_rn(s1.x, t1.x); S[3] = __dsub_rn(s1.y, t1.y);
        }
#pragma unroll
        for (int p = 1; p < BPM_MAX_PAIRS; ++p)
          if (p < npair) {
            const double2 s0 = *reinterpret_cast<const double2*>(pa[p] + i0);
            const double2 s1 = *reinterpret_cast<const double2*>(pa[p] + i0 + 2);
            const double2 t0 = *reinterpret_cast<const double2*>(pb[p] + i0);
            const double2 t1 = *reinterpret_cast<const double2*>(pb[p] + i0 + 2);
            S[0] = __dadd_rn(S[0], __dsub_rn(s0.x, t0.x)); S[1] = __dadd_rn(S[1], __dsub_rn(s0.y, t0.y));
            S[2] = __dadd_rn(S[2], __dsub_rn(s1.x, t1.x)); S[3] = __dadd_rn(S[3], __dsub_rn(s1.y, t1.y));
          }
        double e[4], n[4];
        if (kKeepDraws && dream) {
          e[0] = e[1] = e[2] = e[3] = 0.0;
          n[0] = n[1] = n[2] = n[3] = 0.0;
          if (a.u_eps > 0.0 || a.eps > 0.0) zen_en4(a, qs[kKeepDraws ? t : 0], e, n);
        } else {
          if constexpr (PROB) en4<REPLAY>(a, ps.rng, c, ps.j, b, e, n);
          else en4<REPLAY>(a, c, b, e, n);
        }
        const double cur[4] = {c0.x, c0.y, c1.x, c1.y};
        const double m2v[4] = {w0.x, w0.y, w1.x, w1.y};
        double prv[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int i = i0 + q;
          if (i < a.d) {
            double pr;
            if (dream) {
              const double mf = (mbits >> (4 * t + q)) & 1u ? 1.0 : 0.0;
              pr = dream_prop(cur[q], S[q], e[q], n[q], gamma, mf);
              if (a.adapt) {
                double v;
                if (hist_var) {
                  v = cr_variance<REPLAY>(a, c, i);
                } else {                          // cr_variance's running-moments branch on the preloaded row
                  v = __dmul_rn(m2v[q], a.inv_mom);
                  if (!(v > 0.0)) v = 1e-12 * 1e-12;
                }
                delta += cr_term(cur[q], pr, v);
              }
            } else {
              pr = demc_prop(cur[q], S[q], n[q], gamma);
            }
            prv[q] = pr;
          }
        }
        if (i0 + 3 < a.d) {
          *reinterpret_cast<double2*>(out + i0) = make_double2(prv[0], prv[1]);
          *reinterpret_cast<double2*>(out + i0 + 2) = make_double2(prv[2], prv[3]);
        } else {
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (i0 + q < a.d) out[i0 + q] = prv[q];
        }
        if (a.tr.prop)
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (i0 + q < a.d) a.tr.prop[(size_t)c * a.d + i0 + q] = prv[q];
      }
    }
  } else if (valid) {
#pragma unroll
    for (int t = 0; t < kMaxBlocksPerLane; ++t) {
      const int b = sub + t * LPC;
      if (b < nblk) {
        double e[4], n[4];
        if constexpr (PROB) en4<REPLAY>(a, ps.rng, c, ps.j, b, e, n);
        else en4<REPLAY>(a, c, b, e, n);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int i = 4 * b + q;
          if (i < a.d) {
            const double cur = xc[i];
            double S = __dsub_rn(pa[0][i], pb[0][i]);
#pragma unroll
            for (int p = 1; p < BPM_MAX_PAIRS; ++p)
              if (p < npair) S = __dadd_rn(S, __dsub_rn(pa[p][i], pb[p][i]));
            double pr;
            if (dream) {
              const double mf = (mbits >> (4 * t + q)) & 1u ? 1.0 : 0.0;
              pr = dream_prop(cur, S, e[q], n[q], gamma, mf);
              if (a.adapt) delta += cr_term(cur, pr, cr_variance<REPLAY>(a, c, i));
            } else {
              pr = demc_prop(cur, S, n[q], gamma);
            }
            out[i] = pr;
            if (a.tr.prop) a.tr.prop[(size_t)c * a.d + i] = pr;
          }
        }
      }
    }
  }
  if (dream) {
    delta = group_sum_d<LPC>(delta);
    if (valid && sub == 0) {
      a.cr_pick[c] = a.adapt ? D.cr_idx : -1;
      a.cr_delta[c] = delta;
    }
  }
}

// ---- accept / reject + state, moments, history ---------------------------------
template <bool REPLAY, int LPC, bool PROB = false>
__global__ void __launch_bounds__(kThreads) accept_kernel(const PhaseArgs a, const ProblemArgs prob) {
  const int gid = (blockIdx.x * kThreads + threadIdx.x) / LPC;
  const int sub = threadIdx.x % LPC;
  ProblemSlot ps;
  if constexpr (PROB) ps = problem_slot(a, prob, gid);
  const PhaseLists L = PROB ? slot_lists(ps) : phase_lists(a);
  bool valid = PROB ? ps.valid : gid < L.n_self;
  const int c = PROB ? ps.c : (valid ? L.self[gid] : 0);
  if constexpr (!PROB) valid = valid && c >= a.chain_lo && c < a.chain_hi;
  int acc = 0;
  double lp = 0.0;
  if (valid) {
    lp = a.lnl_prop[gid];
    double u;
    if constexpr (PROB) u = accept_uniform<REPLAY>(a, ps.rng, c, ps.j);
    else u = accept_uniform<REPLAY>(a, c);
    acc = metropolis(a.lnl[c], lp, u);
    if (acc < 0) {
      *a.nan_flag = 1;
      acc = 0;
    }
    double* xc = a.X + (size_t)c * a.ld;
    const double* pr = a.prop + (size_t)gid * a.ld;
    // every array here is per-dimension independent, so the lanes of a chain take CONSECUTIVE
    // dimensions (whole 32-byte sectors per access) instead of the proposal stage's 4-dim blocks
    // (d = 1000 generation 3.34 -> 3.30 ms, gpurun_out/ab10 in profiles/r1_consumer_experiments.txt)
    if (LPC == 32 && ((a.ld | a.d) & 1) == 0) {
      // pairs of consecutive dimensions per lane (16-byte accesses), four pairs per lane loaded before the first
      // store: the scalar loop below cannot overlap an iteration's loads with the previous one's stores (possible
      // aliasing), which left this kernel at 35 % of the DRAM peak at d = 1000
      // (profiles/r2/r2x_c5_propose_accept_ncu.txt).  Same per-dimension arithmetic.
      const size_t ro = (size_t)(c - a.chain_lo) * a.ld;
      const int np2 = a.d >> 1;
      for (int k0 = sub; k0 < np2; k0 += 4 * LPC) {
        double2 sv[4], mu[4], vv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int k = k0 + u * LPC;
          if (k < np2) {
            sv[u] = *reinterpret_cast<const double2*>((acc ? pr : xc) + 2 * k);
            if (a.mean) {
              mu[u] = *reinterpret_cast<const double2*>(a.mean + ro + 2 * k);
              vv[u] = *reinterpret_cast<const double2*>(a.m2 + ro + 2 * k);
            }
          }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int k = k0 + u * LPC;
          if (k < np2) {
            if (acc) {
              *reinterpret_cast<double2*>(xc + 2 * k) = sv[u];
              store_peers2(a, (size_t)c * a.ld + 2 * k, sv[u].x, sv[u].y);
            }
            if (a.mean) {
              welford_update(sv[u].x, a.inv_n1, mu[u].x, vv[u].x);
              welford_update(sv[u].y, a.inv_n1, mu[u].y, vv[u].y);
              *reinterpret_cast<double2*>(a.mean + ro + 2 * k) = mu[u];
              *reinterpret_cast<double2*>(a.m2 + ro + 2 * k) = vv[u];
            }
            if (a.hist_row) *reinterpret_cast<double2*>(a.hist_row + ro + 2 * k) = sv[u];
          }
        }
      }
    } else
#pragma unroll 4
    for (int i = sub; i < a.d; i += LPC) {
      double s = xc[i];
      if (acc) {
        s = pr[i];
        xc[i] = s;
        store_peers1(a, (size_t)c * a.ld + i, s);
      }
      if (a.mean) {  // Welford update with the appended row (chain.py:51-54)
        const size_t o = (size_t)(c - a.chain_lo) * a.ld + i;
        double mu = a.mean[o], v = a.m2[o];
        welford_update(s, a.inv_n1, mu, v);
        a.mean[o] = mu;
        a.m2[o] = v;
      }
      if (a.hist_row) a.hist_row[(size_t)(c - a.chain_lo) * a.ld + i] = s;
    }
    if (sub == 0) {
      if (acc) a.lnl[c] = lp;
      if (a.tr.accept) a.tr.accept[c] = acc;
      if (a.tr.lnl_prop) a.tr.lnl_prop[c] = lp;
    }
  }
  if constexpr (PROB) {
    problem_count(prob, ps.g, valid && sub == 0, acc);
    return;
  }
  const unsigned am = __ballot_sync(0xFFFFFFFFu, valid && sub == 0 && acc);
  const unsigned rm = __ballot_sync(0xFFFFFFFFu, valid && sub == 0 && !acc);
  if ((threadIdx.x & 31) == 0) {
    if (am) atomicAdd(a.n_acc, (unsigned long long)__popc(am));
    if (rm) atomicAdd(a.n_rej, (unsigned long long)__popc(rm));
  }
}

// ---- built-in likelihood kernels over a dense [n][ld] block of rows ---------------
__global__ void lnl_banana_kernel(const double* __restrict__ P, int n, int ld, BananaParams prm,
                                  double* __restrict__ out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) out[j] = banana_lnl(prm, P[(size_t)j * ld], P[(size_t)j * ld + 1]);
}
__global__ void lnl_bimodal_kernel(const double* __restrict__ P, int n, int ld, BimodalParams prm,
                                   double* __restrict__ out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) out[j] = bimodal_lnl(prm, P[(size_t)j * ld], P[(size_t)j * ld + 1]);
}
__global__ void lnl_linefit_kernel(const double* __restrict__ P, int n, int ld,
                                   const double* __restrict__ data, int M, double* __restrict__ out) {
  extern __shared__ double sdata[];
  for (int i = threadIdx.x; i < 3 * M; i += blockDim.x) sdata[i] = data[i];
  __syncthreads();
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n)
    out[j] = linefit_lnl(sdata, sdata + M, sdata + 2 * M, M, P[(size_t)j * ld], P[(size_t)j * ld + 1],
                         P[(size_t)j * ld + 2]);
}

__global__ void lnl_expfit_kernel(const double* __restrict__ P, int n, int ld,
                                  const double* __restrict__ data, int M, double* __restrict__ out) {
  extern __shared__ double sdata[];
  for (int i = threadIdx.x; i < 2 * M; i += blockDim.x) sdata[i] = data[i];
  __syncthreads();
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) {
    const double* th = P + (size_t)j * ld;
    out[j] = expfit_lnl(sdata, sdata + M, M, th[0], th[1], th[2], th[3], th[4]);
  }
}

// Generic tiled quadratic form for any d: out[j] = finish(|(P[j] - mu) . W|^2).
// 64 x 64 output tile per CTA, 4 x 4 register tile per thread, k-tile 16; the tile's
// squared entries are folded into per-row sums so Y = (P - mu) W never reaches memory.
__global__ void __launch_bounds__(256) lnl_gauss_tiled_kernel(const double* __restrict__ P, int n,
                                                              int ld, int d, int r,
                                                              const double* __restrict__ mu,
                                                              const double* __restrict__ W,
                                                              double c0, int log_of_pdf,
                                                              double* __restrict__ out) {
  constexpr int TM = 64, TN = 64, TK = 16;
  __shared__ double As[TK][TM + 1];
  __shared__ double Bs[TK][TN];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.x * TM;
  double rowsum[4] = {0, 0, 0, 0};
  for (int n0 = 0; n0 < r; n0 += TN) {
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.0;
    for (int k0 = 0; k0 < d; k0 += TK) {
      for (int idx = threadIdx.x; idx < TM * TK; idx += 256) {
        const int kk = idx % TK, mm = idx / TK;
        const int row = m0 + mm, k = k0 + kk;
        As[kk][mm] = (row < n && k < d) ? P[(size_t)row * ld + k] - mu[k] : 0.0;
      }
      for (int idx = threadIdx.x; idx < TK * TN; idx += 256) {
        const int nn = idx % TN, kk = idx / TN;
        const int k = k0 + kk, col = n0 + nn;
        Bs[kk][nn] = (k < d && col < r) ? W[(size_t)k * r + col] : 0.0;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < TK; ++kk) {
        double av[4], bv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) av[i] = As[kk][ty * 4 + i];
#pragma unroll
        for (int j = 0; j < 4; ++j) bv[j] = Bs[kk][tx * 4 + j];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fma(av[i], bv[j], acc[i][j]);
      }
      __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) rowsum[i] = fma(acc[i][j], acc[i][j], rowsum[i]);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    double v = rowsum[i];
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    const int row = m0 + ty * 4 + i;
    if (tx == 0 && row < n) out[row] = gauss_finish(c0, v, log_of_pdf);
  }
}

// ---- CR adaptation: deterministic reduction + p_cr update (dream.py:119-140) -----
}  // namespace bpm
#include "cr_reduce.cuh"   // the reduction helpers, shared with the multi-problem CR kernel
namespace bpm {

__global__ void __launch_bounds__(256) cr_update_kernel(const double* __restrict__ cr_delta,
                                                        const int32_t* __restrict__ cr_pick, int lo, int hi,
                                                        int n_cr, double* __restrict__ block_part,
                                                        unsigned int* __restrict__ ticket,
                                                        double* __restrict__ part, int apply,
                                                        double* __restrict__ dm, double* __restrict__ cnt,
                                                        double* __restrict__ p_cr) {
  __shared__ bool last;
  cr_block_partials(cr_delta, cr_pick, lo, hi, n_cr, (int)blockIdx.x, (int)gridDim.x, block_part);
  __threadfence();        // every writer publishes its block partials before the ticket is taken
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (!last) return;
  __threadfence();
  if (threadIdx.x == 0) *ticket = 0u;      // ready for the next generation
  cr_finish(block_part, (int)gridDim.x, n_cr, part, apply, dm, cnt, p_cr);
}

__global__ void cr_apply_kernel(const double* __restrict__ part, int n_cr, double* __restrict__ dm,
                                double* __restrict__ cnt, double* __restrict__ p_cr) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  cr_apply(part, n_cr, dm, cnt, p_cr);
}

// ---- lazy protocol: materialise the pending row (bpm_flush) ---------------------------
// history row hist_len - 1 <- X, and the same row folded into the running moments with the kernels'
// own Welford arithmetic (inv_n = 1 / mom_len: the row is already counted).
__global__ void flush_pending_kernel(const double* __restrict__ X, double* __restrict__ mean,
                                     double* __restrict__ m2, double* __restrict__ hist_cur, int lo, int hi,
                                     int d, int ld, double inv_n) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)(hi - lo) * ld) return;
  const int co = (int)(idx / ld), i = (int)(idx % ld);
  if (i >= d) return;
  const double s = X[(size_t)(lo + co) * ld + i];
  if (mean) {
    double mu = mean[idx], v = m2[idx];
    welford_update(s, inv_n, mu, v);
    mean[idx] = mu;
    m2[idx] = v;
  }
  if (hist_cur) hist_cur[idx] = s;
}

// ---- moments rebuilt from a stored history (load_state / warm start) -------------
__global__ void moments_from_history_kernel(const double* __restrict__ hist, int64_t T, int N, int d,
                                            int ld, int lo, int hi, double* __restrict__ mean,
                                            double* __restrict__ m2) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t tot = (int64_t)(hi - lo) * ld;
  if (idx >= tot) return;
  const int c = lo + (int)(idx / ld), i = (int)(idx % ld);
  if (i >= d) return;
  double mu = 0.0, s2 = 0.0;
  for (int64_t t = 0; t < T; ++t) {
    // the running update of the generation kernels, row by row: a resumed chain gets the
    // moments an uninterrupted one would hold, bit for bit (a column that never moved keeps
    // M2 == 0 exactly, which a two-pass formula does not guarantee)
    const double s = hist[((size_t)t * (hi - lo) + (c - lo)) * ld + i];
    welford_update(s, 1.0 / (double)(t + 1), mu, s2);
  }
  mean[(size_t)(c - lo) * ld + i] = mu;
  m2[(size_t)(c - lo) * ld + i] = s2;
}

// ---- materialise the native stream into replay buffers (testing / provenance) ----
__global__ void dump_draws_kernel(const PhaseArgs a, bpm_replay out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= a.N) return;
  const int c = a.perm[j];
  const bool first_half = j < a.nA;
  const int n_pool = a.serial ? a.N - 1 : (first_half ? a.N - a.nA : a.nA);  // independent of the flip
  const_cast<int32_t*>(out.shuffle_idx)[j] = c;
  ChainDraws D;
  chain_scalar_draws<false>(a, c, n_pool, D);
  const int npair = a.algo == BPM_ALGO_DREAM ? a.del_pairs : 1;
  for (int p = 0; p < npair; ++p) {
    const_cast<int32_t*>(out.pairs)[((size_t)c * npair + p) * 2 + 0] = D.r1[p];
    const_cast<int32_t*>(out.pairs)[((size_t)c * npair + p) * 2 + 1] = D.r2[p];
  }
  const_cast<double*>(out.gamma_u)[c] = D.gamma_u;
  const_cast<double*>(out.accept_u)[c] = accept_uniform<false>(a, c);
  if (a.algo == BPM_ALGO_DREAM) {
    const_cast<int32_t*>(out.cr_idx)[c] = D.cr_idx;
    const_cast<int32_t*>(out.fallback_dim)[c] = D.fallback;
  }
  const int nblk = (a.d + 3) >> 2;
  for (int b = 0; b < nblk; ++b) {
    double z[4], e[4], n[4];
    z4<false>(a, c, b, z);
    en4<false>(a, c, b, e, n);
    for (int q = 0; q < 4; ++q) {
      const int i = 4 * b + q;
      if (i < a.d) {
        if (a.algo == BPM_ALGO_DREAM) {
          const_cast<double*>(out.z)[(size_t)c * a.d + i] = z[q];
          const_cast<double*>(out.e)[(size_t)c * a.d + i] = e[q];
        }
        const_cast<double*>(out.nrm)[(size_t)c * a.d + i] = n[q];
      }
    }
  }
}

}  // namespace bpm
