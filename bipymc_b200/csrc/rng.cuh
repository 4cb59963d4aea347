// Counter-based RNG for the native (non-replay) mode: Philox4x32-10 (Salmon et al.,
// SC'11) written out by hand, plus the counter layout every kernel shares.
//
// The reference draws everything from numpy's global MT19937 stream in chain order
// (demc.py:81,86,169,175; dream.py:51-78; util.py:13,26; samplers.py:336), which is
// inherently serial.  Here every draw is addressed by (seed, absolute generation,
// chain id, purpose, slot), so a chain's step is independent of which thread, tile,
// kernel variant or GPU executes it: a 1-GPU and an 8-GPU run with the same seed make
// the same draws.
#pragma once
#include <stdint.h>

namespace bpm {

struct Philox4 {
  uint32_t x, y, z, w;
};

__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2,
                                                          uint32_t c3, uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = mulhi32(M0, c0), lo0 = M0 * c0;
    uint32_t hi1 = mulhi32(M1, c2), lo1 = M1 * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  Philox4 o = {c0, c1, c2, c3};
  return o;
}

// Purposes (high byte of counter word 3).  The values are part of the counter: renumbering one
// changes the draws of every run that uses it.
enum : uint32_t {
  RNG_SCALAR = 0,  // slot 0: cr_u | accept_u ; slot 1: gamma_u | fallback ; slot 2+p: pair p
  RNG_ZEN = 3,     // slot = dim/4: mask uniform, box jitter and jitter normal of four dims in ONE call
  RNG_GEN = 4,     // chain = 0xFFFFFFFF: slot 0 flip_u + Feistel keys, slot 1 more keys
  RNG_INIT = 5     // device-side chain initialisation jitter
};

struct RngCtx {
  uint32_t k0, k1;  // seed
  uint32_t g_lo;    // absolute generation, low 32 bits
  uint32_t g_hi;    // absolute generation, bits 32..55
};

__host__ __device__ __forceinline__ RngCtx make_rng(uint64_t seed, uint64_t g_abs) {
  RngCtx r;
  r.k0 = (uint32_t)seed;
  r.k1 = (uint32_t)(seed >> 32);
  r.g_lo = (uint32_t)g_abs;
  r.g_hi = (uint32_t)(g_abs >> 32) & 0x00FFFFFFu;
  return r;
}

__host__ __device__ __forceinline__ Philox4 draw4(const RngCtx& r, uint32_t chain, uint32_t purpose,
                                                  uint32_t slot) {
  return philox4x32_10(chain, r.g_lo, slot, (purpose << 24) | r.g_hi, r.k0, r.k1);
}

// [0,1) with 53 random bits, the same grid numpy's random_sample() lives on.
__host__ __device__ __forceinline__ double u53(uint32_t hi, uint32_t lo) {
  uint64_t v = (((uint64_t)hi << 32) | (uint64_t)lo) >> 11;
  return (double)v * (1.0 / 9007199254740992.0);
}
// Unbiased-to-2^-64 integer in [0, n).
__host__ __device__ __forceinline__ uint32_t below64(uint32_t hi, uint32_t lo, uint32_t n) {
  uint64_t v = ((uint64_t)hi << 32) | (uint64_t)lo;
#ifdef __CUDA_ARCH__
  return (uint32_t)__umul64hi(v, (uint64_t)n);
#else
  return (uint32_t)(((unsigned __int128)v * (unsigned __int128)n) >> 64);
#endif
}

#ifdef __CUDACC__
// Two standard normals from 12 + 12 random bits (Box-Muller in fp32: the jitter they feed
// is scaled by epsilon ~ 1e-12, so fp32 shape accuracy is ample).
__device__ __forceinline__ void normal2_12(uint32_t b1, uint32_t b2, float& n0, float& n1) {
  float u1 = ((float)b1 + 1.0f) * (1.0f / 4096.0f);   // (0,1]
  float u2 = (float)b2 * (1.0f / 4096.0f);            // [0,1)
  float r = sqrtf(-2.0f * __logf(u1));
  float s, c;
  __sincosf(6.283185307179586f * u2, &s, &c);
  n0 = r * c;
  n1 = r * s;
}
#endif

// ---------------------------------------------------------------------------------
// Pseudo-random permutation of [0, n) without materialising or sorting anything:
// a balanced Feistel network over 2h >= log2(n) bits with cycle walking.  Replaces
// np.random.shuffle(shuffle_idx) (demc.py:84-86) in native mode; keys come from the
// RNG_GEN stream so every rank derives the same permutation.
struct FeistelKey {
  uint32_t k[6];
  uint32_t half_bits;  // h
  uint32_t n;
};

__host__ __device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
  return x;
}

__host__ __device__ __forceinline__ uint32_t feistel_perm(const FeistelKey& f, uint32_t i) {
  const uint32_t h = f.half_bits, mask = (1u << h) - 1u;
  uint32_t v = i;
  do {
    uint32_t l = v >> h, r = v & mask;
#pragma unroll
    for (int t = 0; t < 6; ++t) {
      uint32_t nl = r;
      r = l ^ (mix32(r ^ f.k[t]) & mask);
      l = nl;
    }
    v = (l << h) | r;
  } while (v >= f.n);
  return v;
}

__host__ __device__ __forceinline__ FeistelKey make_feistel(const RngCtx& r, uint32_t n) {
  FeistelKey f;
  Philox4 a = draw4(r, 0xFFFFFFFFu, RNG_GEN, 1), b = draw4(r, 0xFFFFFFFFu, RNG_GEN, 2);
  f.k[0] = a.x; f.k[1] = a.y; f.k[2] = a.z; f.k[3] = a.w; f.k[4] = b.x; f.k[5] = b.y;
  uint32_t bits = 1;
  while ((1ull << bits) < (unsigned long long)n) ++bits;
  f.half_bits = (bits + 1) / 2;
  if (f.half_bits == 0) f.half_bits = 1;
  f.n = n;
  return f;
}

}  // namespace bpm
