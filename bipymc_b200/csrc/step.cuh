// Shared device-side pieces of one DE-MC / DREAM chain-step: kernel parameter block,
// draw providers (native Philox or RNG-replay), and the proposal / accept arithmetic
// written with explicit round-to-nearest intrinsics so the compiler can never contract
// a multiply-add -- in replay mode the proposal must reproduce numpy's elementwise
// float64 results bit for bit (demc.py:180-182, dream.py:85-89).
#pragma once
#include <stdint.h>
#include "rng.cuh"
#include "../../include/bipymc_b200.h"

// compute-sanitizer is closed on the GPU pool this was developed on (profiles/r2/r2e_sanitizer_*.log), so the
// index checks it would have made are built in: -DBPM_CHECKS=1 turns every chain / partner / list index of the
// phase kernels into a checked access that prints and traps (tools/sanitize_case.py runs all kernel families
// under such a build; the shipped library compiles the checks away).
#ifndef BPM_CHECKS
#define BPM_CHECKS 0
#endif
#if BPM_CHECKS
#include <stdio.h>
#define BPM_CHECK(cond, what, v)                                                                          \
  do {                                                                                                   \
    if (!(cond)) {                                                                                       \
      printf("BPM_CHECK failed: %s = %lld (%s:%d, block %d thread %d)\n", what, (long long)(v), __FILE__,  \
             __LINE__, (int)blockIdx.x, (int)threadIdx.x);                                               \
      __trap();                                                                                          \
    }                                                                                                    \
  } while (0)
#else
#define BPM_CHECK(cond, what, v) do { } while (0)
#endif

namespace bpm {

// Everything a phase kernel needs, passed by value (fits the 4 KB param space easily).
struct PhaseArgs {
  // population (caller-owned)
  double* X;
  double* lnl;
  double* mean;
  double* m2;
  double* hist_row;  // destination row block [n_local][ld] for this generation, or nullptr (eager kernels)
  // lazy protocol (fused_gauss_v3_kernel): the kernel does NOT append the new state to the history /
  // running moments; it leaves that row pending and folds the row the PREVIOUS generation left pending
  // -- each chain's current state, which its proposal stage holds in registers anyway -- instead.
  double* hist_cur;  // history row hist_len - 1 (the pending one) [n_local][ld], or nullptr
  int32_t lazy;      // this launch follows the lazy protocol
  int32_t pending;   // the current row of every chain is not yet in mean / m2 / history: fold it now
  const double* hist_base;  // row 0 of the stored history (replay mode: exact np.std), or nullptr
  // phase lists: perm[0:nA) is half "a", perm[nA:N) half "b" before the flip swap
  const int32_t* perm;
  const int32_t* flip;  // device flag (demc.py:81,98-100)
  // The flag is a function of (seed, generation) -- or the replayed value -- so the host evaluates it too and
  // passes it by value: the kernels' first dependent global load (flag -> list -> chain id -> rows) goes away.
  int32_t flip_known;   // flip_val below is valid
  // sharded handles: this rank's chains of each half, compacted in list order into
  // loc_list[0 : loc_cnt[0]) and loc_list[nA : nA + loc_cnt[1]); nullptr when the rank owns all chains
  const int32_t* loc_list;
  const int32_t* loc_cnt;
  int32_t phase;        // 0: update a from frozen b; 1: update b from updated a
  int32_t N, nA, d, ld;
  int32_t chain_lo, chain_hi;
  // schedule
  int32_t algo, del_pairs, n_cr;
  int32_t serial;      // BPM_ALGO_DEMC_SERIAL: self = every chain, pool = every OTHER chain
  int32_t gamma_jump;  // k % 5 == 0 (DREAM, dream.py:77) / k % 10 == 0 (DE-MC, demc.py:174)
  double gamma_p0;     // 0.2 / 0.1: probability of KEEPING gamma_base on a jump generation
  double gamma_fixed;  // DE-MC gamma_base (demc.py:162)
  double gamma_num;    // DREAM: gamma_scale * 2.38 (dream.py:61)
  double eps;          // Gaussian jitter sd (already sqrt(epsilon**2))
  double u_eps;        // box jitter half-width
  int32_t adapt;       // burnin_gen > k && hist_len > n_cr_gen (dream.py:92,124)
  int64_t hist_len;    // rows in every chain's history BEFORE this generation's append
  int64_t mom_len;     // rows covered by the running moments BEFORE this generation
  double inv_mom;      // 1 / mom_len
  double inv_n1;       // 1 / (mom_len + 1)
  // CR state
  const double* p_cr;  // [n_cr]
  double* cr_delta;    // [N] per-chain jump statistic of this generation (or untouched)
  int32_t* cr_pick;    // [N] chosen CR index, -1 when no statistic was recorded
  // workspace
  double* prop;      // [nA][ld] proposals in phase order
  double* lnl_prop;  // [nA]
  // peer replicas of X on the other GPUs (bpm_set_peers); accepted rows are stored there too
  double* peers[BPM_MAX_PEERS];
  int32_t n_peers;
  // counters
  unsigned long long* n_acc;
  unsigned long long* n_rej;
  int32_t* nan_flag;
  int32_t flip_val;     // the flip flag's value (host_flip or the replayed coin), valid when flip_known
  // native RNG
  RngCtx rng;
  // replay buffers (REPLAY kernels only)
  bpm_replay rp;
  // optional trace
  bpm_trace_out tr;
};

// Accepted row -> every peer replica (4 doubles of chain c starting at element off; 16-byte aligned).
__device__ __forceinline__ void store_peers4(const PhaseArgs& a, size_t elem_off, double s0, double s1,
                                             double s2, double s3) {
  for (int p = 0; p < a.n_peers; ++p) {
    double* q = a.peers[p] + elem_off;
    *reinterpret_cast<double2*>(q) = make_double2(s0, s1);
    *reinterpret_cast<double2*>(q + 2) = make_double2(s2, s3);
  }
}
__device__ __forceinline__ void store_peers2(const PhaseArgs& a, size_t elem_off, double s0, double s1) {
  for (int p = 0; p < a.n_peers; ++p) *reinterpret_cast<double2*>(a.peers[p] + elem_off) = make_double2(s0, s1);
}
__device__ __forceinline__ void store_peers1(const PhaseArgs& a, size_t elem_off, double s) {
  for (int p = 0; p < a.n_peers; ++p) a.peers[p][elem_off] = s;
}

// Phase-list helpers.  self = chains updated in this phase, pool = the other half.
struct PhaseLists {
  const int32_t* self;
  const int32_t* pool;
  int32_t n_self, n_pool;
  int32_t skip_self;   // pool position r of chain c means chain r + (r >= c): np.delete(range(N), c)[r]
};
// global chain id of pool position r for the chain c being stepped
__device__ __forceinline__ int pool_chain(const PhaseLists& L, int r, int c) {
  BPM_CHECK(r >= 0 && r < L.n_pool, "pool position", r);
  return L.skip_self ? r + (r >= c ? 1 : 0) : L.pool[r];
}
__device__ __forceinline__ PhaseLists phase_lists(const PhaseArgs& a) {
  const int32_t first = (a.phase ^ (a.flip_known ? a.flip_val : (*a.flip != 0))) == 0;  // true: self is perm[0:nA)
  PhaseLists L;
  L.skip_self = 0;
  if (a.serial) {   // samplers.py:275-277: valid_pool_ids = np.delete(range(n_chains), i)
    L.self = a.perm; L.n_self = a.N; L.pool = a.perm; L.n_pool = a.N - 1; L.skip_self = 1;
    if (a.loc_cnt) { L.self = a.loc_list; L.n_self = a.loc_cnt[0]; }
    return L;
  }
  if (first) {
    L.self = a.perm; L.n_self = a.nA; L.pool = a.perm + a.nA; L.n_pool = a.N - a.nA;
  } else {
    L.self = a.perm + a.nA; L.n_self = a.N - a.nA; L.pool = a.perm; L.n_pool = a.nA;
  }
  if (a.loc_cnt) {   // only the local chains of the half, densely packed
    L.self = a.loc_list + (first ? 0 : a.nA);
    // (a handle that owns every chain packs whole halves: the counts are known without the load)
    L.n_self = (a.chain_lo == 0 && a.chain_hi == a.N) ? (first ? a.nA : a.N - a.nA) : a.loc_cnt[first ? 0 : 1];
  }
  return L;
}

// ---- multi-problem handles (bpm_set_problems) --------------------------------------
// P independent populations of n chains each, problem-major: problem g owns chains [g n, (g + 1) n).  Each
// has its own Philox key, flip, a/b split, CR state and counters, so problem g steps exactly as a handle of
// n chains with key keys[g] would.  The split kernel (kernels_problems.cuh) writes, per problem, the halves
// in permutation order to perm[g n, g n + nA) / [g n + nA, (g + 1) n) (global chain ids) and the same halves
// in chain order to loc_list.  Thread t of a phase kernel steps slot t % nA of problem t / nA's half.
struct ProblemArgs {
  const uint64_t* keys;            // [P] Philox key of each problem
  const int32_t* flips;            // [P] this generation's flip of each problem
  const double* p_cr;              // [P][BPM_MAX_CR]
  unsigned long long* counters;    // [P][2] accepted, rejected
  int32_t P, n, nA;                // problems, chains per problem, ceil(n / 2)
};
// What a phase kernel needs of the chain at slot t: its global id c, its index j within the problem (the
// RNG counter a single-problem handle uses for it), the pool of the opposite half and the problem's key.
struct ProblemSlot {
  int g, c, j, n_pool;
  bool valid;
  const int32_t* pool;
  RngCtx rng;
  const double* p_cr;
};
__device__ __forceinline__ ProblemSlot problem_slot(const PhaseArgs& a, const ProblemArgs& pb, int t) {
  ProblemSlot s;
  s.g = t / pb.nA;
  const int i = t - s.g * pb.nA;
  s.valid = s.g < pb.P;
  if (!s.valid) s.g = 0;
  const int base = s.g * pb.n;
  const bool first = (a.phase ^ (pb.flips[s.g] != 0)) == 0;   // true: this phase steps half a
  const int n_self = first ? pb.nA : pb.n - pb.nA;
  s.valid = s.valid && i < n_self;
  s.c = s.valid ? a.loc_list[base + (first ? 0 : pb.nA) + i] : base;
  s.j = s.c - base;
  s.pool = a.perm + base + (first ? pb.nA : 0);
  s.n_pool = first ? pb.n - pb.nA : pb.nA;
  s.rng = make_rng(pb.keys[s.g], (uint64_t)a.hist_len);
  s.p_cr = pb.p_cr + (size_t)s.g * BPM_MAX_CR;
  return s;
}
// Per-problem accepted / rejected counts of a warp: one atomic per problem the warp touches.
__device__ __forceinline__ void problem_count(const ProblemArgs& pb, int g, bool valid, int acc) {
  const unsigned same = __match_any_sync(0xFFFFFFFFu, g);
  const unsigned am = __ballot_sync(0xFFFFFFFFu, valid && acc) & same;
  const unsigned rm = __ballot_sync(0xFFFFFFFFu, valid && !acc) & same;
  if ((threadIdx.x & 31) == __ffs(same) - 1) {
    if (am) atomicAdd(pb.counters + 2 * g, (unsigned long long)__popc(am));
    if (rm) atomicAdd(pb.counters + 2 * g + 1, (unsigned long long)__popc(rm));
  }
}

// Reduce over the LPC lanes that share one chain (LPC is a power of two <= 32).
template <int LPC>
__device__ __forceinline__ int group_sum_i(int v) {
#pragma unroll
  for (int o = LPC / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  return v;
}
template <int LPC>
__device__ __forceinline__ double group_sum_d(double v) {
#pragma unroll
  for (int o = LPC / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  return v;
}

// numpy choice over a cdf: idx = searchsorted(cdf / cdf[-1], u, side='right')
// (legacy RandomState.choice; dream.py:51).
__device__ __forceinline__ int pick_cr(const double* p_cr, int n_cr, double u) {
  double tot = 0.0;
  for (int m = 0; m < n_cr; ++m) tot = __dadd_rn(tot, p_cr[m]);
  double acc = 0.0;
  int idx = 0;
  for (int m = 0; m < n_cr; ++m) {
    acc = __dadd_rn(acc, p_cr[m]);
    if (__ddiv_rn(acc, tot) <= u) idx = m + 1;
  }
  return idx < n_cr ? idx : n_cr - 1;
}

// samplers.py:328-336: alpha = clip(min(1, exp(lp - lc)), 0, 1);
// accept iff u < alpha / (alpha + (1 - alpha))   (numpy choice with p=[alpha, 1-alpha]).
// Returns 1 accept, 0 reject, -1 NaN alpha (numpy raises ValueError there).
__device__ __forceinline__ int metropolis(double lnl_cur, double lnl_prop, double u) {
  double alpha = exp(__dsub_rn(lnl_prop, lnl_cur));
  if (alpha != alpha) return -1;
  alpha = alpha > 1.0 ? 1.0 : alpha;
  alpha = alpha < 0.0 ? 0.0 : alpha;
  double thr = __ddiv_rn(alpha, __dadd_rn(alpha, __dsub_rn(1.0, alpha)));
  return u < thr ? 1 : 0;
}

// Per-chain scalar draws.
struct ChainDraws {
  int cr_idx;
  int fallback;
  double gamma_u;
  int r1[BPM_MAX_PAIRS], r2[BPM_MAX_PAIRS];  // POOL-LOCAL partner indices
};

// Layout of the per-chain scalar stream RNG_SCALAR (one Philox call per slot):
//   slot 0   words x,y -> uniform behind the CR choice   | z,w -> uniform behind accept
//   slot 1   words x,y -> uniform behind the gamma choice | z,w -> fallback dimension
//   slot 2+p pair p: x,y -> first partner, z,w -> second partner (distinct, ordered:
//            the law of np.random.permutation(P)[:2], demc.py:169 / dream.py:66)
__device__ __forceinline__ double slot0_cr_u(const Philox4& q) { return u53(q.x, q.y); }
__device__ __forceinline__ double slot0_accept_u(const Philox4& q) { return u53(q.z, q.w); }
__device__ __forceinline__ double slot1_gamma_u(const Philox4& q) { return u53(q.x, q.y); }
__device__ __forceinline__ int slot1_fallback(const Philox4& q, int d) {
  return (int)below64(q.z, q.w, (uint32_t)d);
}
__device__ __forceinline__ void slot_pair(const Philox4& q, int n_pool, int& r1, int& r2) {
  uint32_t i = below64(q.x, q.y, (uint32_t)n_pool);
  uint32_t j = below64(q.z, q.w, (uint32_t)(n_pool - 1));
  j += (j >= i);
  r1 = (int)i;
  r2 = (int)j;
}

// The draws of chain c are addressed by (rng, j): j = c on a single-problem handle; on a multi-problem
// handle rng carries the problem's key and j is the chain's index within its problem (ProblemArgs).
template <bool REPLAY>
__device__ __forceinline__ void chain_scalar_draws(const PhaseArgs& a, const RngCtx& rng, const double* p_cr, int c,
                                                   int j, int n_pool, ChainDraws& D) {
  const int npair = a.algo == BPM_ALGO_DREAM ? a.del_pairs : 1;
  if (REPLAY) {
    D.cr_idx = a.algo == BPM_ALGO_DREAM ? a.rp.cr_idx[c] : 0;
    D.fallback = a.algo == BPM_ALGO_DREAM ? a.rp.fallback_dim[c] : -1;
    D.gamma_u = a.rp.gamma_u[c];
#pragma unroll
    for (int p = 0; p < BPM_MAX_PAIRS; ++p)
      if (p < npair) {
        D.r1[p] = a.rp.pairs[((size_t)c * npair + p) * 2 + 0];
        D.r2[p] = a.rp.pairs[((size_t)c * npair + p) * 2 + 1];
      }
  } else {
    const Philox4 s0 = draw4(rng, (uint32_t)j, RNG_SCALAR, 0);
    const Philox4 s1 = draw4(rng, (uint32_t)j, RNG_SCALAR, 1);
    D.cr_idx = a.algo == BPM_ALGO_DREAM ? pick_cr(p_cr, a.n_cr, slot0_cr_u(s0)) : 0;
    D.gamma_u = slot1_gamma_u(s1);
    D.fallback = slot1_fallback(s1, a.d);
#pragma unroll
    for (int p = 0; p < BPM_MAX_PAIRS; ++p)
      if (p < npair) slot_pair(draw4(rng, (uint32_t)j, RNG_SCALAR, 2 + p), n_pool, D.r1[p], D.r2[p]);
  }
}
template <bool REPLAY>
__device__ __forceinline__ void chain_scalar_draws(const PhaseArgs& a, int c, int n_pool, ChainDraws& D) {
  chain_scalar_draws<REPLAY>(a, a.rng, a.p_cr, c, c, n_pool, D);
}

template <bool REPLAY>
__device__ __forceinline__ double accept_uniform(const PhaseArgs& a, const RngCtx& rng, int c, int j) {
  if (REPLAY) return a.rp.accept_u[c];
  return slot0_accept_u(draw4(rng, (uint32_t)j, RNG_SCALAR, 0));
}
template <bool REPLAY>
__device__ __forceinline__ double accept_uniform(const PhaseArgs& a, int c) {
  return accept_uniform<REPLAY>(a, a.rng, c, c);
}

// The three per-dimension draws of a 4-dim block -- crossover-mask uniform z (dream.py:52), box jitter e
// (dream.py:83) and jitter normal n (dream.py:84) -- come from ONE Philox call (purpose RNG_ZEN, slot b).
// Word k of the call belongs to dim 4b + k:  bits 0-11 z on a 4096-point grid, bits 12-19 e on a 256-point
// grid, bits 20-31 twelve bits towards a Box-Muller pair (words 0,1 -> n0,n1; words 2,3 -> n2,n3).
// The mask compares z with CR in {1/n_cr ..}: a 2^-12 grid moves each crossover probability by < 2.5e-4;
// e only randomises gamma by +-1 %; n has sd epsilon ~ 1e-12.  A chain-step of the fused kernel is bound by
// its instruction count, and a Philox call is ~70 of ~850 (profiles/r2c_*).
// Measured (profiles/r2d_*): 125.7 -> 118.0 us per launch of the fused 100-D kernel against two calls per
// block (32-bit z, 16-bit e, 16 + 16-bit Box-Muller).
__device__ __forceinline__ void zen_z4(const Philox4& q, double z[4]) {
  z[0] = ((double)(q.x & 0xFFFu) + 0.5) * (1.0 / 4096.0); z[1] = ((double)(q.y & 0xFFFu) + 0.5) * (1.0 / 4096.0);
  z[2] = ((double)(q.z & 0xFFFu) + 0.5) * (1.0 / 4096.0); z[3] = ((double)(q.w & 0xFFFu) + 0.5) * (1.0 / 4096.0);
}
__device__ __forceinline__ uint32_t zen_mask4(const Philox4& q, uint32_t th12) {
  return ((q.x & 0xFFFu) <= th12 ? 1u : 0u) | ((q.y & 0xFFFu) <= th12 ? 2u : 0u) |
         ((q.z & 0xFFFu) <= th12 ? 4u : 0u) | ((q.w & 0xFFFu) <= th12 ? 8u : 0u);
}
// u = (z12 + 0.5) / 4096 <= cr  <=>  z12 <= floor(cr * 4096 - 0.5)
__device__ __forceinline__ uint32_t zen_threshold(double cr) {
  const double lim = floor(cr * 4096.0 - 0.5);
  return lim >= 4095.0 ? 0xFFFu : (lim < 0.0 ? 0xFFFFFFFFu : (uint32_t)lim);   // lim < 0: nothing passes (wraps: never <=)
}
__device__ __forceinline__ void zen_en4(const PhaseArgs& a, const Philox4& q, double e[4], double n[4]) {
  e[0] = e[1] = e[2] = e[3] = 0.0;
  n[0] = n[1] = n[2] = n[3] = 0.0;
  if (a.u_eps > 0.0) {
    const double lo = -a.u_eps, w = __dsub_rn(a.u_eps, lo);
    const double w9 = w * (1.0 / 512.0);           // (h + 0.5) / 256 = (2h + 1) / 512
    e[0] = __dadd_rn(lo, __dmul_rn(w9, (double)(int)(2u * ((q.x >> 12) & 0xFFu) + 1u)));
    e[1] = __dadd_rn(lo, __dmul_rn(w9, (double)(int)(2u * ((q.y >> 12) & 0xFFu) + 1u)));
    e[2] = __dadd_rn(lo, __dmul_rn(w9, (double)(int)(2u * ((q.z >> 12) & 0xFFu) + 1u)));
    e[3] = __dadd_rn(lo, __dmul_rn(w9, (double)(int)(2u * ((q.w >> 12) & 0xFFu) + 1u)));
  }
  if (a.eps > 0.0) {
    float f0, f1, f2, f3;
    normal2_12(q.x >> 20, q.y >> 20, f0, f1);
    normal2_12(q.z >> 20, q.w >> 20, f2, f3);
    n[0] = __dmul_rn(a.eps, (double)f0);
    n[1] = __dmul_rn(a.eps, (double)f1);
    n[2] = __dmul_rn(a.eps, (double)f2);
    n[3] = __dmul_rn(a.eps, (double)f3);
  }
}

// Four per-dimension draws for dims 4b .. 4b+3 of chain c.
template <bool REPLAY>
__device__ __forceinline__ void z4(const PhaseArgs& a, const RngCtx& rng, int c, int j, int b, double z[4]) {
  if (REPLAY) {
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      int i = 4 * b + t;
      z[t] = i < a.d ? a.rp.z[(size_t)c * a.d + i] : 2.0;
    }
  } else {
    zen_z4(draw4(rng, (uint32_t)j, RNG_ZEN, (uint32_t)b), z);
  }
}
template <bool REPLAY>
__device__ __forceinline__ void z4(const PhaseArgs& a, int c, int b, double z[4]) {
  z4<REPLAY>(a, a.rng, c, c, b, z);
}
// Box jitter e (dream.py:83, var_box) and Gaussian jitter n (demc.py:182 / dream.py:84,
// var_ball) for dims 4b .. 4b+3, from the block's RNG_ZEN call (zen_en4).
template <bool REPLAY>
__device__ __forceinline__ void en4(const PhaseArgs& a, const RngCtx& rng, int c, int j, int b, double e[4],
                                    double n[4]) {
  if (REPLAY) {
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      int i = 4 * b + t;
      e[t] = (i < a.d && a.rp.e) ? a.rp.e[(size_t)c * a.d + i] : 0.0;
      n[t] = (i < a.d && a.rp.nrm) ? a.rp.nrm[(size_t)c * a.d + i] : 0.0;
    }
  } else {
    e[0] = e[1] = e[2] = e[3] = 0.0;  // var_box returns 0. and draws nothing (util.py:24-28)
    n[0] = n[1] = n[2] = n[3] = 0.0;  // var_ball returns 0. and draws nothing (util.py:11-16)
    if (a.u_eps > 0.0 || a.eps > 0.0) zen_en4(a, draw4(rng, (uint32_t)j, RNG_ZEN, (uint32_t)b), e, n);
  }
}

template <bool REPLAY>
__device__ __forceinline__ void en4(const PhaseArgs& a, int c, int b, double e[4], double n[4]) {
  en4<REPLAY>(a, a.rng, c, c, b, e, n);
}

// dream.py:85-89:  ((1 + e) * gamma * S + n) * mask + cur, evaluated left to right.
__device__ __forceinline__ double dream_prop(double cur, double S, double e, double n, double gamma,
                                             double maskf) {
  double t = __dadd_rn(1.0, e);
  t = __dmul_rn(t, gamma);
  t = __dmul_rn(t, S);
  t = __dadd_rn(t, n);
  t = __dmul_rn(t, maskf);
  return __dadd_rn(t, cur);
}
// demc.py:180-182:  gamma * (a - b); += cur; += n
__device__ __forceinline__ double demc_prop(double cur, double diff, double n, double gamma) {
  double t = __dmul_rn(gamma, diff);
  t = __dadd_rn(t, cur);
  return __dadd_rn(t, n);
}

// dream.py:61 / 77-80 and demc.py:162 / 174-177
__device__ __forceinline__ double dream_gamma(const PhaseArgs& a, int d_prime, double gamma_u) {
  double base = __ddiv_rn(a.gamma_num, __dsqrt_rn(__dmul_rn(__dmul_rn(2.0, (double)a.del_pairs),
                                                            (double)d_prime)));
  if (a.gamma_jump) return gamma_u < a.gamma_p0 ? base : 1.0;
  return base;
}
__device__ __forceinline__ double demc_gamma(const PhaseArgs& a, double gamma_u) {
  if (a.gamma_jump) return gamma_u < a.gamma_p0 ? a.gamma_fixed : 1.0;
  return a.gamma_fixed;
}

// dream.py:128-129: std_devs = np.std(chain.chain, axis=0); std_devs[std_devs == 0] = 1e-12;
// returns std_devs ** 2 for dimension i of chain c.
//   native mode : running (Welford) moments, var = M2 / T, O(1) per step;
//   replay mode : numpy's own two-pass algorithm over the stored history column
//                 (sequential sums along axis 0, mean = sum / T, var = sum((x - mean)^2) / T,
//                 sqrt, then squared again), O(T) per step.  This matters for parity: for a
//                 column that never moved np.std returns rounding noise (~1e-17 * |x|)
//                 instead of 0, the reference's `== 0` guard does not fire, and the
//                 chain's jump statistic is divided by ~1e-34.  Replay reproduces that
//                 to the bit; native mode gets an exact 0 and the 1e-12 floor.
template <bool REPLAY>
__device__ __forceinline__ double cr_variance(const PhaseArgs& a, int c, int i) {
  const int co = c - a.chain_lo;
  if (REPLAY && a.hist_base != nullptr) {
    const size_t stride = (size_t)(a.chain_hi - a.chain_lo) * a.ld;
    const double* p = a.hist_base + (size_t)co * a.ld + i;
    const double T = (double)a.hist_len;
    double sum = p[0];
    for (int64_t t = 1; t < a.hist_len; ++t) sum = __dadd_rn(sum, p[t * stride]);
    const double mean = __ddiv_rn(sum, T);
    double ss = 0.0;
    for (int64_t t = 0; t < a.hist_len; ++t) {
      const double dx = __dsub_rn(p[t * stride], mean);
      ss = __dadd_rn(ss, __dmul_rn(dx, dx));
    }
    double sd = __dsqrt_rn(__ddiv_rn(ss, T));
    if (sd == 0.0) sd = 1e-12;
    return __dmul_rn(sd, sd);
  }
  double var = __dmul_rn(a.m2[(size_t)co * a.ld + i], a.inv_mom);
  if (!(var > 0.0)) var = 1e-12 * 1e-12;
  return var;
}

// Reciprocal to ~1 ulp without the IEEE division's slow path: hardware seed + two Newton
// steps.  Only the CR jump statistic uses it (a sum over thousands of chains that is
// compared with the reference to 1e-10), never the chain arithmetic itself.
__device__ __forceinline__ double fast_rcp(double v) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(v));
  double e = fma(-v, r, 1.0);
  r = fma(r, e, r);
  e = fma(-v, r, 1.0);
  r = fma(r, e, r);
  return r;
}

// dream.py:130 contribution of one dimension: (cur - prop)^2 / std^2.
__device__ __forceinline__ double cr_term(double cur, double prop, double var) {
  const double df = __dsub_rn(cur, prop);
  if (df == 0.0) return 0.0;               // dimensions outside the crossover subspace
  const double sq = __dmul_rn(df, df);
  const double r = fast_rcp(var);
  if (!(r > 0.0) || !(r < 1.7e308)) return __ddiv_rn(sq, var);   // var = inf / denormal / NaN
  return __dmul_rn(sq, r);
}

// Explicitly rounded Welford update (identical bits in every kernel that uses it).
__device__ __forceinline__ void welford_update(double s, double inv_n1, double& mu, double& m2) {
  const double dl = __dsub_rn(s, mu);
  const double mu2 = __dadd_rn(mu, __dmul_rn(dl, inv_n1));   // inv_n1 = 1 / (rows + 1), from the host
  m2 = __dadd_rn(m2, __dmul_rn(dl, __dsub_rn(s, mu2)));
  mu = mu2;
}

}  // namespace bpm
