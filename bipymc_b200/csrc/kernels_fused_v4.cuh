// fused_gauss_v4_kernel -- the fused Gaussian half-phase with the chain-pair gathers STAGED THROUGH
// SHARED MEMORY BY TMA (demc.py:153-196, dream.py:32-107 for half of the population in one launch).
//
// Why (profiles/r2a_lazy_v3_fused_gauss_ncu_summary.txt, profiles/r2_gather_probe2_b200.txt): in v3 a
// producer warp gathers a chain's 2 * del_pairs partner rows with LDG.128 into 48 landing registers and
// sits on the long scoreboard for ~1.3 us before it can start ~2.5 us of dependent arithmetic (39 % of
// all warp-state samples).  A fair probe shows cp.async.bulk row copies sustain 6.7 - 8.2 TB/s when every
// warp issues them, so the gather does not have to occupy a warp at all.  Here
//   * every producer warp owns ONE landing slot of 2 * del_pairs rows in shared memory.  The slot is busy
//     only from the copy's issue until the pair differences S are summed -- the first ~50 ns of a
//     chain's arithmetic -- so the gather of chain n+1 is issued right after S of chain n and runs under
//     the rest of chain n (Philox draws, crossover mask, jitter, proposal, lazy moments update);
//   * the chain's own row and M2 row (sequential, streamed) are prefetched into 16 registers at the same
//     moment -- registers the landing area no longer needs; the mean row is loaded once S is done;
//   * the landing slots (16 x 4.8 KB at d = 100) take the shared memory of v3's second proposal tile:
//     there is ONE 64-row proposal tile, handed over per 8-row m-tile (named barrier per m-tile towards
//     the consumer -- a blocking hardware wait, no polling -- and mbarrier DONEm[8] back); a producer
//     writes its row of m-tile cw only after consumer cw released the previous tile's;
//   * consumers are v3's: 8 warps, one m-tile each on the FP64 tensor pipe (mma.sync.m8n8k4.f64, W in
//     DMMA fragment order in shared memory), Metropolis decision in registers, accepted rows stored from
//     the tile (and into the peer replicas) by the deciding warp.
// Lazy protocol as v3 (PhaseArgs::pending).  Draw values and proposal arithmetic are every other
// path's (same helpers), so chains are bit-identical to v3's.
#pragma once
#include "kernels_fused.cuh"

namespace bpm {

__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_addr(dst)), "l"(src), "r"(bytes), "r"(smem_addr(bar)) : "memory");
}

// Accepted row -> own replica and every peer replica as TMA bulk copies straight out of the proposal tile:
// one instruction per destination (1 + n_peers of them) from ONE lane, asynchronous -- instead of two 16-byte
// stores per lane per destination that the deciding warp has to push through its own store path (at 8 GPUs the
// peer stores cost 17 us of a 141 us launch, profiles/r2/r2k_bench_n8_nopeerstores.json).
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               ::"l"(dst), "r"(smem_addr(src_smem)), "r"(bytes) : "memory");
}

struct V4Layout {
  size_t wf, mus, gam, cdf, crv, thr, P, acc_u, cid, land, scratch, bars, total;   // byte offsets
  int land_rows;
};
__host__ __device__ inline V4Layout v4_layout(int d, int r, int npair) {
  V4Layout L;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += (bytes + 127) & ~(size_t)127; return at; };
  L.wf = take(sizeof(double) * (size_t)(d >> 2) * dmma_ntiles(r) * 32);
  L.mus = take(sizeof(double) * d);
  L.gam = take(sizeof(double) * (d + 1));
  L.cdf = take(sizeof(double) * BPM_MAX_CR);
  L.crv = take(sizeof(double) * BPM_MAX_CR);
  L.thr = take(sizeof(uint32_t) * BPM_MAX_CR);
  L.P = take(sizeof(double) * (size_t)kTileRows * dmma_pld(d));
  L.acc_u = take(sizeof(double) * kTileRows);
  L.cid = take(sizeof(int) * kTileRows);
  L.land_rows = 2 * npair;
  L.land = take(sizeof(double) * (size_t)kV3ProdWarps * L.land_rows * d);
  L.scratch = take(2 * ((sizeof(TileScratch) + 127) & ~(size_t)127));
  L.bars = take(sizeof(uint64_t) * (kV3ProdWarps + 2 * kV3ConsWarps));     // LAND[16], DONEm[8], WREADY, 7 spare
  L.total = o;
  return L;
}
inline bool fused_v4_fits(int d, int ld, int r, int npair) {
  return (d % 4) == 0 && ld == d && npair >= 1 && npair <= BPM_MAX_PAIRS && 2 * npair <= 32 &&
         v4_layout(d, r, npair).total <= kMaxDynSmem;
}

constexpr int kV4BarFull0 = 3;                       // named barriers 3 .. 10 (0 = __syncthreads, 2 = BAR_CONS)
constexpr int kV4FullCount = 32 * (8 + 1);           // 8 producing warps + the consumer warp

// rows of the own chain prefetched one chain ahead
struct V4Pre {
  double2 u0, u1, w0, w1;
  int c;
};

template <bool REPLAY, bool CENTER, int NPAIR>
__global__ void __launch_bounds__(kV3Threads, 1)
fused_gauss_v4_kernel(const PhaseArgs a, const GaussArgs g) {
  extern __shared__ __align__(128) unsigned char smem4[];
  const int d = a.d, pld = dmma_pld(d), NT = dmma_ntiles(g.r);
  // NPAIR = 3: DREAM with three pairs, NPAIR = 1: DE-MC (one pair, no crossover / CR statistics), both resolved at
  // compile time; NPAIR = 0: algorithm and pair count read from the arguments
  const bool dream = NPAIR == 3 ? true : (NPAIR == 1 ? false : a.algo == BPM_ALGO_DREAM);
  const int npair = NPAIR == 3 ? 3 : (NPAIR == 1 ? 1 : (dream ? a.del_pairs : 1));
  const V4Layout L4 = v4_layout(d, g.r, npair);
  GaussTables tb;
  tb.Ws = reinterpret_cast<double*>(smem4 + L4.wf);
  tb.mus = reinterpret_cast<double*>(smem4 + L4.mus);
  tb.gam = reinterpret_cast<double*>(smem4 + L4.gam);
  tb.cdf = reinterpret_cast<double*>(smem4 + L4.cdf);
  tb.crv = reinterpret_cast<double*>(smem4 + L4.crv);
  tb.thr = reinterpret_cast<uint32_t*>(smem4 + L4.thr);
  double* P = reinterpret_cast<double*>(smem4 + L4.P);
  double* row_u = reinterpret_cast<double*>(smem4 + L4.acc_u);     // accept uniform of every tile row
  int* row_c = reinterpret_cast<int*>(smem4 + L4.cid);             // chain id of every tile row, -1 = empty
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem4 + L4.bars);
  uint64_t* LAND = bars;                               // [16] partner rows of the warp's chain have landed
  uint64_t* DONEm = bars + kV3ProdWarps;               // [8]  consumer cw is done with its m-tile
  uint64_t* WREADY = DONEm + kV3ConsWarps;             // W fragments + mu have landed (TMA, g.Wf != nullptr)
  // "all 8 rows of m-tile cw are in the tile" is named barrier kV4BarFull0 + cw: 8 producing warps arrive,
  // the consumer warp syncs
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int w = 0; w < kV3ProdWarps; ++w) mbar_init(LAND + w, 1);
    for (int w = 0; w < kV3ConsWarps; ++w) mbar_init(DONEm + w, 1);
    mbar_init(WREADY, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (g.Wf) {
      // W (83 KB at d = r = 100, fragment order prepared by w_fragment_kernel) and mu arrive as two bulk copies
      // issued before anything else happens in the CTA; the consumers wait for them on WREADY.  The in-kernel
      // rearrangement this replaces (load_W_fragments) held the consumer warps for the first ~20 us of a launch:
      // 6.3 % of all warp samples on its one load line, profiles/r2/r2zd_v4_source_lines.txt.
      const uint32_t wbytes = (uint32_t)(sizeof(double) * (size_t)(d >> 2) * NT * 32), mbytes = (uint32_t)(d * 8);
      mbar_expect_tx(WREADY, wbytes + mbytes);
      bulk_g2s(tb.Ws, g.Wf, wbytes, WREADY);
      bulk_g2s(tb.mus, g.mu, mbytes, WREADY);
    }
  }
  fill_tables_v3(a, g, tb, threadIdx.x, kV3Threads);
  __syncthreads();
  const PhaseLists L = phase_lists(a);
  const int per_cta = (L.n_self + (int)gridDim.x - 1) / (int)gridDim.x;
  const int g_lo = min((int)blockIdx.x * per_cta, L.n_self);
  const int g_hi = min(g_lo + per_cta, L.n_self);
  const int n_my = (g_hi - g_lo + kTileRows - 1) / kTileRows;

  if (warp < kV3ConsWarps) {
    // ------------------------------ consumers ------------------------------------------
    asm volatile("setmaxnreg.dec.sync.aligned.u32 64;");
    if (g.Wf) {
      mbar_wait(WREADY, 0);
    } else {
      load_W_fragments(tb.Ws, tb.mus, g.W, g.mu, d, g.r, threadIdx.x, kV3ConsThreads);
      nbar_sync(BAR_CONS, kV3ConsThreads);
    }
    unsigned n_acc = 0, n_rej = 0;
    const bool decider = (lane & 3) == 0;
    const int my_row = 8 * warp + (lane >> 2);
    for (int i = 0; i < n_my; ++i) {
      nbar_sync(kV4BarFull0 + warp, kV4FullCount);      // blocks until the 8 producing warps arrived
      const double maha = gauss_tile_maha_dmma8<CENTER>(P, pld, tb.Ws, tb.mus, d, NT, warp, lane);
      const int c = decider ? row_c[my_row] : -1;
      int acc = 0;
      if (c >= 0) {
        const double lp = gauss_finish(g.c0, maha, g.log_of_pdf);
        acc = metropolis(a.lnl[c], lp, row_u[my_row]);
        if (acc < 0) {
          *a.nan_flag = 1;
          acc = 0;
        }
        if (acc) a.lnl[c] = lp;
        if (a.tr.accept) a.tr.accept[c] = acc;
        if (a.tr.lnl_prop) a.tr.lnl_prop[c] = lp;
      }
      unsigned am = __ballot_sync(0xFFFFFFFFu, c >= 0 && acc);
      n_acc += __popc(am);
      n_rej += __popc(__ballot_sync(0xFFFFFFFFu, c >= 0 && !acc));
      if (am) {                                      // ~1 accepted row per m-tile
        if (lane == 0) {
          // the rows were written through the generic proxy (producers' st.shared, ordered by the named barrier)
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          const uint32_t row_bytes = (uint32_t)(d * 8);
          while (am) {
            const int row = 8 * warp + ((__ffs(am) - 1) >> 2);
            am &= am - 1;
            const size_t ox = (size_t)row_c[row] * a.ld;
            const double* src = P + row * pld;
            bulk_s2g(a.X + ox, src, row_bytes);
            for (int p = 0; p < a.n_peers; ++p) bulk_s2g(a.peers[p] + ox, src, row_bytes);
          }
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the tile rows have been read
        }
        __syncwarp();
      }
      if (lane == 0) mbar_arrive(DONEm + warp);      // (lane 0's tile reads, the last of the warp's, are done)
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // every row has reached memory
    if (lane == 0) {
      if (n_acc) atomicAdd(a.n_acc, (unsigned long long)n_acc);
      if (n_rej) atomicAdd(a.n_rej, (unsigned long long)n_rej);
    }
    return;
  }

  // ------------------------------ producers --------------------------------------------
  asm volatile("setmaxnreg.inc.sync.aligned.u32 88;");
  const int pw = warp - kV3ConsWarps;
  if (n_my == 0) return;
  const size_t t_stride = (sizeof(TileScratch) + 127) & ~(size_t)127;
  auto scratch = [&](int tile) -> TileScratch& {
    return *reinterpret_cast<TileScratch*>(smem4 + L4.scratch + (size_t)(tile & 1) * t_stride);
  };
  double* land = reinterpret_cast<double*>(smem4 + L4.land) + (size_t)pw * L4.land_rows * d;
  // Lanes past the row (4 lane >= d; 7 of 32 at d = 100) do the work of the last real lane on the same
  // addresses and simply never store: no divergence, no zero-filled stand-in values.
  const bool act = 4 * lane < d;
  const int lc = act ? lane : (d >> 2) - 1;
  const bool adapt = dream && a.adapt;
  const bool welford_var = adapt && !(REPLAY && a.hist_base != nullptr);
  const bool fold = a.pending && a.mean != nullptr;
  const bool need_m2 = fold || welford_var;
  const uint32_t land_bytes = (uint32_t)(2 * npair * d * 8);
  const int n_total = 4 * n_my;                  // this warp's chains: tile i, rows pw + 16 j
  uint32_t land_phase = 0;

  // gather of chain n: TMA copies of its partner rows into the landing slot + register prefetch of its own rows
  auto start_chain = [&](int n, V4Pre& pre) {
    const TileScratch& T = scratch(n >> 2);
    const int row = pw + kV3ProdWarps * (n & 3);
    const int c = T.cid[row];
    pre.c = c;
    if (c < 0) return;
    if (lane == 0) mbar_expect_tx(LAND + pw, land_bytes);
    __syncwarp();
    if (lane < 2 * npair) {
      const int p = lane >> 1;
      const int id = (lane & 1) ? T.pb[row][p] : T.pa[row][p];
      BPM_CHECK(id >= 0 && id < a.N, "partner chain id (TMA source row)", id);
      BPM_CHECK((size_t)((lane + 1) * d) <= (size_t)L4.land_rows * d, "landing slot row", lane);
      bulk_g2s(land + (size_t)lane * d, a.X + (size_t)id * a.ld, (uint32_t)(d * 8), LAND + pw);
    }
    BPM_CHECK(c >= a.chain_lo && c < a.chain_hi, "own chain id", c);
    const double* xc = a.X + (size_t)c * a.ld + 4 * lc;
    pre.u0 = ldg2(xc); pre.u1 = ldg2(xc + 2);
    if (need_m2) {
      const double* mp = a.m2 + (size_t)(c - a.chain_lo) * a.ld + 4 * lc;
      pre.w0 = ld_stream2(mp); pre.w1 = ld_stream2(mp + 2);
    }
  };
  // row `row` of the tile is complete: all 32 lanes arrive on the m-tile's named barrier (the consumer
  // blocks in bar.sync there -- a hardware wait that costs no issue slots, unlike an mbarrier poll)
  auto hand_over = [&](int i, int row, int cw, int c, double u, const double* prv) {
    BPM_CHECK(row >= 0 && row < kTileRows && cw == (row >> 3), "tile row", row);
    if (i >= 1) mbar_wait(DONEm + cw, (i - 1) & 1);     // consumer cw released tile i-1's m-tile
    if (act) {
      double* prow = P + row * pld + 4 * lane;
      *reinterpret_cast<double2*>(prow) = make_double2(prv[0], prv[1]);
      *reinterpret_cast<double2*>(prow + 2) = make_double2(prv[2], prv[3]);
    }
    if (lane == 0) {
      row_c[row] = c;
      row_u[row] = u;
    }
    nbar_arrive(kV4BarFull0 + cw, kV4FullCount);
  };

  warp_stage_draws<REPLAY>(a, L, tb, scratch(0), g_lo, g_hi, pw, lane);
  V4Pre pre;
  pre.u0 = pre.u1 = pre.w0 = pre.w1 = make_double2(0.0, 0.0);
  start_chain(0, pre);
#pragma unroll 1
  for (int n = 0; n < n_total; ++n) {
    const int i = n >> 2, j = n & 3;
    const int row = pw + kV3ProdWarps * j, cw = row >> 3;
    if (j == 0 && i + 1 < n_my)      // draws one tile ahead; scratch (i+1)&1 was tile i-1's, and this warp is through with it
      warp_stage_draws<REPLAY>(a, L, tb, scratch(i + 1), g_lo + (i + 1) * kTileRows, g_hi, pw, lane);
    const TileScratch& T = scratch(i);
    const int c = pre.c;
    if (c < 0) {                     // past the end of this CTA's range (last tile only): an empty row
      const double zero[4] = {0.0, 0.0, 0.0, 0.0};
      if (n + 1 < n_total) start_chain(n + 1, pre);
      hand_over(i, row, cw, -1, 0.0, zero);
      continue;
    }
    double cur[4] = {pre.u0.x, pre.u0.y, pre.u1.x, pre.u1.y};
    double var[4] = {pre.w0.x, pre.w0.y, pre.w1.x, pre.w1.y};
    double S[4];
    mbar_wait(LAND + pw, land_phase & 1);
    land_phase += 1;
    {
      const double* lp = land + 4 * lc;
      if constexpr (NPAIR == 3) {
        double2 va[3][2], vb[3][2];
#pragma unroll
        for (int p = 0; p < 3; ++p) {
          va[p][0] = *reinterpret_cast<const double2*>(lp + (2 * p) * d);
          va[p][1] = *reinterpret_cast<const double2*>(lp + (2 * p) * d + 2);
          vb[p][0] = *reinterpret_cast<const double2*>(lp + (2 * p + 1) * d);
          vb[p][1] = *reinterpret_cast<const double2*>(lp + (2 * p + 1) * d + 2);
        }
        S[0] = __dsub_rn(va[0][0].x, vb[0][0].x); S[1] = __dsub_rn(va[0][0].y, vb[0][0].y);
        S[2] = __dsub_rn(va[0][1].x, vb[0][1].x); S[3] = __dsub_rn(va[0][1].y, vb[0][1].y);
#pragma unroll
        for (int p = 1; p < 3; ++p) {
          S[0] = __dadd_rn(S[0], __dsub_rn(va[p][0].x, vb[p][0].x));
          S[1] = __dadd_rn(S[1], __dsub_rn(va[p][0].y, vb[p][0].y));
          S[2] = __dadd_rn(S[2], __dsub_rn(va[p][1].x, vb[p][1].x));
          S[3] = __dadd_rn(S[3], __dsub_rn(va[p][1].y, vb[p][1].y));
        }
      } else {
        S[0] = S[1] = S[2] = S[3] = 0.0;
        for (int p = 0; p < npair; ++p) {
          const double2 s0 = *reinterpret_cast<const double2*>(lp + (2 * p) * d);
          const double2 s1 = *reinterpret_cast<const double2*>(lp + (2 * p) * d + 2);
          const double2 t0 = *reinterpret_cast<const double2*>(lp + (2 * p + 1) * d);
          const double2 t1 = *reinterpret_cast<const double2*>(lp + (2 * p + 1) * d + 2);
          const double df0 = __dsub_rn(s0.x, t0.x), df1 = __dsub_rn(s0.y, t0.y);
          const double df2 = __dsub_rn(s1.x, t1.x), df3 = __dsub_rn(s1.y, t1.y);
          S[0] = p == 0 ? df0 : __dadd_rn(S[0], df0);
          S[1] = p == 0 ? df1 : __dadd_rn(S[1], df1);
          S[2] = p == 0 ? df2 : __dadd_rn(S[2], df2);
          S[3] = p == 0 ? df3 : __dadd_rn(S[3], df3);
        }
      }
    }
    __syncwarp();                                                       // every lane has read the slot ...
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // ... before the async proxy refills it
    // the next chain's gather runs under the rest of this chain
    if (n + 1 < n_total) start_chain(n + 1, pre);

    const size_t o = (size_t)(c - a.chain_lo) * a.ld + 4 * lc;
    double2 mn0 = make_double2(0.0, 0.0), mn1 = mn0;
    if (a.pending) {
      // the mean row's latency hides behind the draws below; the pending history row leaves from registers
      if (fold) { mn0 = ld_stream2(a.mean + o); mn1 = ld_stream2(a.mean + o + 2); }
      if (a.hist_cur && act) {
        st_stream2(a.hist_cur + o, cur[0], cur[1]);
        st_stream2(a.hist_cur + o + 2, cur[2], cur[3]);
      }
    }
    uint32_t mbits = 0xFu;
    double gamma;
    const double gu = T.gamma_u[row];
    Philox4 qzen = {0u, 0u, 0u, 0u};       // the block's single Philox call, shared by the mask and the jitters
    if (dream) {
      const int m = T.cr_idx[row];
      if (REPLAY) {
        const double cr = tb.crv[m];
        double z[4];
        z4<REPLAY>(a, c, lc, z);
        mbits = (z[0] <= cr ? 1u : 0u) | (z[1] <= cr ? 2u : 0u) | (z[2] <= cr ? 4u : 0u) | (z[3] <= cr ? 8u : 0u);
      } else {
        const uint32_t th = tb.thr[m];
        qzen = draw4(a.rng, (uint32_t)c, RNG_ZEN, (uint32_t)lc);
        mbits = zen_mask4(qzen, th);
      }
      int d_prime = __reduce_add_sync(0xFFFFFFFFu, act ? __popc(mbits) : 0);
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
    double delta = 0.0, prv[4];
    {
      double e[4], nn[4];
      if (!REPLAY && dream) zen_en4(a, qzen, e, nn);
      else en4<REPLAY>(a, c, lc, e, nn);
      if (fold) {
        welford_update(cur[0], a.inv_mom, mn0.x, var[0]);
        welford_update(cur[1], a.inv_mom, mn0.y, var[1]);
        welford_update(cur[2], a.inv_mom, mn1.x, var[2]);
        welford_update(cur[3], a.inv_mom, mn1.y, var[3]);
        if (act) {
          st_stream2(a.mean + o, mn0.x, mn0.y); st_stream2(a.mean + o + 2, mn1.x, mn1.y);
          st_stream2(a.m2 + o, var[0], var[1]); st_stream2(a.m2 + o + 2, var[2], var[3]);
        }
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
              v = cr_variance<REPLAY>(a, c, 4 * lc + q);
            }
            delta += cr_term(cur[q], pr, v);
          }
        } else {
          pr = demc_prop(cur[q], S[q], nn[q], gamma);
        }
        prv[q] = pr;
      }
      if (REPLAY && a.tr.prop && act) {
        double* tp = a.tr.prop + (size_t)c * d + 4 * lane;
#pragma unroll
        for (int q = 0; q < 4; ++q) tp[q] = prv[q];
      }
    }
    if (dream) {
      delta = group_sum_d<32>(act ? delta : 0.0);
      if (lane == 0) {
        a.cr_pick[c] = adapt ? T.cr_idx[row] : -1;
        a.cr_delta[c] = delta;
      }
    }
    hand_over(i, row, cw, c, T.accept_u[row], prv);
  }
}

template <bool REPLAY, bool CENTER, int NPAIR>
inline int launch_fused_v4(const PhaseArgs& a, const GaussArgs& g, int grid, size_t sm, cudaStream_t s) {
  cudaError_t e = cudaFuncSetAttribute(fused_gauss_v4_kernel<REPLAY, CENTER, NPAIR>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
  if (e != cudaSuccess) return 1;
  fused_gauss_v4_kernel<REPLAY, CENTER, NPAIR><<<grid, kV3Threads, sm, s>>>(a, g);
  return 0;
}

}  // namespace bpm
