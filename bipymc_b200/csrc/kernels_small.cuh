// d <= 4 targets, one thread per chain: the chain-step shared by every d <= 4 kernel and the per-phase
// fused_small_kernel.  Device code only: besides the engine build, the run-time compiled likelihoods
// (BPM_TARGET_JIT, engine.cu: bpm_jit_compile) compile this header with NVRTC, which has no host runtime.
//
// BPM_JIT_LIKELIHOOD is defined only by that NVRTC translation unit, which places the user's
//   __device__ double ln_like(const double* theta, const double* data)
// before this header; the engine build never refers to ln_like.
#pragma once
#include "step.cuh"
#include "targets.cuh"

namespace bpm {

struct TargetView {
  int target;
  BananaParams banana;
  BimodalParams bimodal;
  const double* mu;
  const double* W;
  const double* Wf;   // see GaussArgs
  int r;
  double c0;
  int log_of_pdf;
  int mu_is_zero;
  const double* linefit;
  int linefit_M;
  const double* data;     // BPM_TARGET_JIT: the user likelihood's data array (device), n_data doubles
  int64_t n_data;
};

// BPM_TARGET_JIT: data arrays of up to this many doubles (32 KB) are staged in the kernels' dynamic shared
// memory, larger ones are read from global memory (where L1 / L2 hold them: every thread reads the same values).
constexpr int64_t kJitSmemDoubles = 4096;

// ---- d <= 4 analytic targets: one thread per chain ------------------------------------
// One chain-step of a d <= 4 target, start to finish (draws, proposal, likelihood, Metropolis decision,
// state / moments / history update).  pool_id(r) maps a pool position to a global chain id: a lookup in the
// materialised shuffle for the per-phase kernel, the Feistel permutation evaluated on the fly for the
// persistent multi-generation kernel.  Returns 1 when the proposal was accepted.
template <bool REPLAY, int TARGET, typename PoolFn>
__device__ __forceinline__ int small_chain_step(const PhaseArgs& a, const TargetView& tv, const double* sdata,
                                                int c, int n_pool, PoolFn pool_id) {
  const int d = a.d;
  const bool dream = a.algo == BPM_ALGO_DREAM;
  const int npair = dream ? a.del_pairs : 1;
  ChainDraws D;
  chain_scalar_draws<REPLAY>(a, c, n_pool, D);
  BPM_CHECK(c >= a.chain_lo && c < a.chain_hi, "own chain id", c);
  for (int p = 0; p < npair; ++p) {
    BPM_CHECK(D.r1[p] >= 0 && D.r1[p] < n_pool && D.r2[p] >= 0 && D.r2[p] < n_pool && D.r1[p] != D.r2[p],
              "pair draw", D.r1[p] * 100000LL + D.r2[p]);
    BPM_CHECK(pool_id(D.r1[p]) >= 0 && pool_id(D.r1[p]) < a.N && pool_id(D.r2[p]) >= 0 && pool_id(D.r2[p]) < a.N,
              "partner chain id", pool_id(D.r1[p]));
  }
  uint32_t mbits = 0xFu;
  double gamma;
  if (dream) {
    mbits = 0u;
    const double cr = __ddiv_rn((double)(D.cr_idx + 1), (double)a.n_cr);
    double z[4];
    z4<REPLAY>(a, c, 0, z);
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (q < d && z[q] <= cr) mbits |= 1u << q;
    int d_prime = __popc(mbits);
    if (d_prime == 0) {
      mbits |= 1u << ((D.fallback < 0 ? 0 : D.fallback) & 3);
      d_prime = 1;
    }
    gamma = dream_gamma(a, d_prime, D.gamma_u);
  } else {
    gamma = demc_gamma(a, D.gamma_u);
  }
  double* xc = a.X + (size_t)c * a.ld;
  double cur[4] = {0, 0, 0, 0}, S[4] = {0, 0, 0, 0}, pr[4] = {0, 0, 0, 0};
  // Everything the step reads of its OWN chain is requested here, in one batch of independent loads: the
  // cached likelihood and the moments rows would otherwise each cost an exposed round trip AFTER the likelihood
  // (the stores in between keep the compiler from hoisting them; ncu: long scoreboard 27 % of the line-fit
  // kernel's warp time, profiles/r2/r2x_fused_small_linefit_ncu_summary.txt).
  // Only where one chain-step is long and few warps are resident (the line fit): on the 2-D targets the twelve
  // extra registers cost a resident block per SM (94 -> 106 registers; 10^6 bimodal chains: 0.22 -> 0.27 ms per
  // generation, profiles/r2/r2y_secondary.txt), so those load late as before.
  constexpr bool kPreload = TARGET == BPM_TARGET_LINEFIT || TARGET == BPM_TARGET_JIT;
  double mu_c[4] = {0, 0, 0, 0}, m2_c[4] = {0, 0, 0, 0};
  double lnl_c = 0.0;
  if constexpr (kPreload) {
    const size_t o = (size_t)(c - a.chain_lo) * a.ld;
    lnl_c = a.lnl[c];
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (q < d) {
        cur[q] = xc[q];
        if (a.mean) {
          mu_c[q] = a.mean[o + q];
          m2_c[q] = a.m2[o + q];
        }
      }
  } else {
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (q < d) cur[q] = xc[q];
  }
#pragma unroll
  for (int p = 0; p < BPM_MAX_PAIRS; ++p)
    if (p < npair) {
      const double* pa = a.X + (size_t)pool_id(D.r1[p]) * a.ld;
      const double* pb = a.X + (size_t)pool_id(D.r2[p]) * a.ld;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (q < d) {
          const double df = __dsub_rn(pa[q], pb[q]);
          S[q] = p == 0 ? df : __dadd_rn(S[q], df);
        }
    }
  double e[4], nn[4];
  en4<REPLAY>(a, c, 0, e, nn);
  double delta = 0.0;
#pragma unroll
  for (int q = 0; q < 4; ++q)
    if (q < d) {
      if (dream) {
        pr[q] = dream_prop(cur[q], S[q], e[q], nn[q], gamma, (mbits >> q) & 1u ? 1.0 : 0.0);
        if constexpr (kPreload) {
          if (a.adapt) {
            double v;
            if ((REPLAY && a.hist_base != nullptr) || !a.mean) {
              v = cr_variance<REPLAY>(a, c, q);
            } else {                             // cr_variance's running-moments branch on the preloaded row
              v = __dmul_rn(m2_c[q], a.inv_mom);
              if (!(v > 0.0)) v = 1e-12 * 1e-12;
            }
            delta += cr_term(cur[q], pr[q], v);
          }
        } else {
          if (a.adapt) delta += cr_term(cur[q], pr[q], cr_variance<REPLAY>(a, c, q));
        }
      } else {
        pr[q] = demc_prop(cur[q], S[q], nn[q], gamma);
      }
    }
  if (dream) {
    a.cr_pick[c] = a.adapt ? D.cr_idx : -1;
    a.cr_delta[c] = delta;
  }
  if (REPLAY && a.tr.prop)
#pragma unroll
    for (int q = 0; q < 4; ++q)
      if (q < d) a.tr.prop[(size_t)c * d + q] = pr[q];
  double lp;
  if (TARGET == BPM_TARGET_BANANA) lp = banana_lnl(tv.banana, pr[0], pr[1]);
  else if (TARGET == BPM_TARGET_BIMODAL) lp = bimodal_lnl(tv.bimodal, pr[0], pr[1]);
#ifdef BPM_JIT_LIKELIHOOD
  else if constexpr (TARGET == BPM_TARGET_JIT) lp = ln_like(pr, tv.n_data <= kJitSmemDoubles ? sdata : tv.data);
#endif
  else lp = linefit_lnl(sdata, sdata + tv.linefit_M, sdata + 2 * tv.linefit_M, tv.linefit_M, pr[0],
                        pr[1], pr[2]);
  int acc;
  if constexpr (kPreload) acc = metropolis(lnl_c, lp, accept_uniform<REPLAY>(a, c));
  else acc = metropolis(a.lnl[c], lp, accept_uniform<REPLAY>(a, c));
  if (acc < 0) {
    *a.nan_flag = 1;
    acc = 0;
  }
  const size_t o = (size_t)(c - a.chain_lo) * a.ld;
#pragma unroll
  for (int q = 0; q < 4; ++q)
    if (q < d) {
      const double s = acc ? pr[q] : cur[q];
      if (acc) {
        xc[q] = s;
        store_peers1(a, (size_t)c * a.ld + q, s);
      }
      if (a.mean) {
        double mu, v;
        if constexpr (kPreload) { mu = mu_c[q]; v = m2_c[q]; }
        else { mu = a.mean[o + q]; v = a.m2[o + q]; }
        welford_update(s, a.inv_n1, mu, v);
        a.mean[o + q] = mu;
        a.m2[o + q] = v;
      }
      if (a.hist_row) a.hist_row[o + q] = s;
    }
  if (acc) a.lnl[c] = lp;
  if (a.tr.accept) a.tr.accept[c] = acc;
  if (a.tr.lnl_prop) a.tr.lnl_prop[c] = lp;
  return acc;
}

template <bool REPLAY, int TARGET>
__global__ void __launch_bounds__(128) fused_small_kernel(const PhaseArgs a, const TargetView tv) {
  extern __shared__ __align__(16) double sdata[];
  if (TARGET == BPM_TARGET_LINEFIT) {
    for (int i = threadIdx.x; i < 3 * tv.linefit_M; i += blockDim.x) sdata[i] = tv.linefit[i];
    __syncthreads();
  }
#ifdef BPM_JIT_LIKELIHOOD
  if constexpr (TARGET == BPM_TARGET_JIT) {
    if (tv.n_data <= kJitSmemDoubles) {
      for (int i = threadIdx.x; i < tv.n_data; i += blockDim.x) sdata[i] = tv.data[i];
      __syncthreads();
    }
  }
#endif
  const PhaseLists L = phase_lists(a);
  const int gid = blockIdx.x * blockDim.x + threadIdx.x;
  bool valid = gid < L.n_self;
  const int c = valid ? L.self[gid] : 0;
  valid = valid && c >= a.chain_lo && c < a.chain_hi;
  int acc = 0;
  if (valid) acc = small_chain_step<REPLAY, TARGET>(a, tv, sdata, c, L.n_pool, [&](int r) { return L.pool[r]; });
  const unsigned am = __ballot_sync(0xFFFFFFFFu, valid && acc);
  const unsigned rm = __ballot_sync(0xFFFFFFFFu, valid && !acc);
  if ((threadIdx.x & 31) == 0) {
    if (am) atomicAdd(a.n_acc, (unsigned long long)__popc(am));
    if (rm) atomicAdd(a.n_rej, (unsigned long long)__popc(rm));
  }
}

#ifdef BPM_JIT_LIKELIHOOD
// ln_like over a dense [n][ld] block of rows, one thread per row (split path, serial DE-MC, bpm_eval_lnl).
__global__ void __launch_bounds__(128) lnl_jit_kernel(const double* __restrict__ P, int n, int ld,
                                                      const double* __restrict__ data, int64_t n_data,
                                                      double* __restrict__ out) {
  extern __shared__ __align__(16) double sdata[];
  const double* dp = data;
  if (n_data <= kJitSmemDoubles) {
    for (int i = threadIdx.x; i < n_data; i += blockDim.x) sdata[i] = data[i];
    __syncthreads();
    dp = sdata;
  }
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) out[j] = ln_like(P + (size_t)j * ld, dp);
}
#endif

}  // namespace bpm
