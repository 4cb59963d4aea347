// Multi-problem handles (bpm_set_problems, step.cuh: ProblemArgs): the per-problem split.  Their phase kernels are
// the PROB branches of propose_kernel / accept_kernel (kernels_generic.cuh) and of the run-time compiled chain-step
// (kernels_small.cuh, BPM_JIT_PROBLEMS); their CR reduction is cr_update_problems_kernel (cr_reduce.cuh), compiled
// into the same run-time module.
#pragma once
#include "kernels_generic.cuh"

namespace bpm {

constexpr int kSplitThreads = 128;

// One CTA per problem g.  What split_native_kernel and the list-compaction kernels produce on a handle of n
// chains with key keys[g]: the flip coin and the Feistel keys from RNG_GEN (chain 0xFFFFFFFF) of that key,
// perm[g n + i] = g n + feistel(i) (the halves in permutation order: pools), and the same halves in chain
// order in loc_list (the chains a phase steps, so that their rows are read in ascending order).  inv is
// scratch: inv[g n + c] = position of chain c in the problem's permutation.
__global__ void __launch_bounds__(kSplitThreads) split_problems_kernel(int32_t* __restrict__ perm,
                                                                       int32_t* __restrict__ inv,
                                                                       int32_t* __restrict__ loc_list,
                                                                       int32_t* __restrict__ flips, int n, int nA,
                                                                       int shuffle, double flip_p,
                                                                       const uint64_t* __restrict__ keys,
                                                                       uint64_t g_abs) {
  const int g = blockIdx.x;
  const int base = g * n;
  __shared__ FeistelKey fkey;
  if (threadIdx.x == 0) {
    const RngCtx rng = make_rng(keys[g], g_abs);
    const Philox4 q = draw4(rng, 0xFFFFFFFFu, RNG_GEN, 0);
    const double thr = __ddiv_rn(flip_p, __dadd_rn(flip_p, __dsub_rn(1.0, flip_p)));
    flips[g] = u53(q.x, q.y) < thr ? 1 : 0;
    if (shuffle) fkey = make_feistel(rng, (uint32_t)n);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += kSplitThreads) {
    const int c = shuffle ? (int)feistel_perm(fkey, (uint32_t)i) : i;
    perm[base + i] = base + c;
    inv[base + c] = i;
  }
  __syncthreads();     // makes the block's inv stores visible to the whole block
  int offA = 0, offB = 0;
  for (int c0 = 0; c0 < n; c0 += kSplitThreads) {
    const int c = c0 + threadIdx.x;
    const int inA = c < n && inv[base + c] < nA ? 1 : 0;
    const int inB = c < n && !inA ? 1 : 0;
    int ea, eb, ta, tb;
    block_excl_scan2<kSplitThreads>(inA, inB, ea, eb, ta, tb);
    if (inA) loc_list[base + offA + ea] = base + c;
    if (inB) loc_list[base + nA + offB + eb] = base + c;
    offA += ta;
    offB += tb;
    __syncthreads();   // the scan's shared totals are read above before the next chunk overwrites them
  }
}

}  // namespace bpm
