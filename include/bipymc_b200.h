/*
 * bipymc_b200 -- C-ABI of the B200-native DE-MC / DREAM generation engine.
 *
 * Drop-in boundary for the per-generation hot path of wgurecky/bipymc.  Every entry
 * point names the reference interface it replaces (paths relative to the reference
 * repo).  Plain pointers and sizes only; no C++ or torch types cross this boundary.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; bpm_last_error()
 *     returns a thread-local message for the last failure.  No C++ exception escapes.
 *   - "device pointer" = CUDA device memory on the handle's device, owned by the
 *     CALLER (the Python host keeps them in torch tensors).  The library only borrows
 *     them for the duration of a call (kernels are enqueued on `stream`; the caller
 *     synchronises).  Library-owned memory is limited to the opaque handle's workspace.
 *   - population layout: X[n_chains][ld] float64, chain-major rows, ld >= dim, rows
 *     16-byte aligned.  lnl[n_chains] caches ln_like(X[c]).
 *   - one host thread per handle at a time.
 */
#ifndef BIPYMC_B200_H_
#define BIPYMC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BPM_ALGO_DEMC 0   /* DeMcMpi._update_chain_pool   bipymc/demc.py:153-196 */
#define BPM_ALGO_DREAM 1  /* DreamMpi._update_chain_pool  bipymc/dream.py:32-107 */
#define BPM_ALGO_DEMC_SERIAL 2 /* DeMc._mcmc_run, delayed accept: every chain proposes from the frozen
                                  population, partners drawn from ALL other chains, no a/b split, no
                                  gamma jumps (bipymc/samplers.py:261-308); one phase per generation */

#define BPM_MAX_PAIRS 8
#define BPM_MAX_CR 16
#define BPM_MAX_PEERS 15

/* Built-in batched likelihoods (the reference's test targets, SURVEY.md section 8a L1-L4). */
#define BPM_TARGET_EXTERNAL 0 /* ln_like supplied through bpm_propose / bpm_accept or a callback */
#define BPM_TARGET_BANANA 1   /* bipymc/utils/banana_rv.py:26-37   params: bpm_mvn2 + a, b        */
#define BPM_TARGET_BIMODAL 2  /* bipymc/utils/dblgauss_rv.py:26-32 params: 2 x bpm_mvn2 + weights  */
#define BPM_TARGET_GAUSS 3    /* bipymc/utils/d100_gauss.py:14-35  params: mu[d], W[d][r], c0      */
#define BPM_TARGET_LINEFIT 4  /* examples/ex_para_fit.py:39-55     params: x[M], y[M], yerr[M]     */
#define BPM_TARGET_EXPFIT 5   /* examples/ex_exp_fit.py:38-121     params: t[M], y[M]; dim = 5     */
#define BPM_TARGET_JIT 6      /* user CUDA source compiled at run time: bpm_set_jit_target only   */
#define BPM_TARGET_JIT_SUM 7  /* per-observation CUDA source, summed: bpm_set_jit_sum_target only */

typedef struct bpm_engine* bpm_handle;
typedef void* bpm_stream; /* cudaStream_t */

/* Sampler configuration = the ctor / run_mcmc kwargs of the reference
 * (demc.py:14-27,73-75,161-162; dream.py:17-27,40-41). */
typedef struct bpm_config {
  int32_t algo;       /* BPM_ALGO_*                                               */
  int32_t n_chains;   /* N, global population size (>= 4, samplers.py:249)        */
  int32_t dim;        /* d                                                        */
  int32_t ld;         /* row stride of X / history / moments in doubles           */
  int32_t del_pairs;  /* DREAM pairs per proposal (dream.py:22), 1 for DE-MC      */
  int32_t n_cr;       /* number of crossover values (dream.py:27)                 */
  int32_t burnin_gen; /* CR adaptation runs while burnin_gen > k (dream.py:24,92) */
  int32_t n_cr_gen;   /* ... and once len(chain) > n_cr_gen (dream.py:26,124)     */
  int32_t shuffle;    /* run_mcmc(shuffle=...) demc.py:74                         */
  int32_t chain_lo;   /* this rank owns chains [chain_lo, chain_hi)  (demc.py:39) */
  int32_t chain_hi;
  int32_t device;     /* CUDA device ordinal                                      */
  double gamma_scale; /* dream.py:20                                              */
  double flip;        /* run_mcmc(flip=...) demc.py:73, already clipped to [0,1]  */
  double epsilon;     /* Gaussian jitter sd (demc.py:161 1e-15, dream.py:40 1e-12)*/
  double u_epsilon;   /* DREAM uniform jitter half-width (dream.py:41)            */
  double gamma;       /* DE-MC jump rate (demc.py:162); <= 0 selects 2.38/sqrt(2d)*/
  uint64_t seed;      /* Philox key (native-RNG mode)                             */
} bpm_config;

/* Caller-owned device arrays the generation step reads and updates in place. */
typedef struct bpm_state {
  double* X;        /* [n_chains][ld]  current positions of the WHOLE population (every rank
                       keeps a replica; rows outside [chain_lo, chain_hi) are read-only
                       partner states refreshed by the host's all-gather)              */
  double* lnl;      /* [n_chains]      cached ln_like(X[c]); only the local rows are used */
  /* the arrays below cover only this rank's chains, n_local = chain_hi - chain_lo,
     indexed by (c - chain_lo): */
  double* mean;     /* [n_local][ld]   running mean of each chain's history, or NULL    */
  double* m2;       /* [n_local][ld]   running sum of squared deviations, or NULL       */
  double* history;  /* [>= hist_len + n_gen][n_local][ld] or NULL: row t = state after
                       generation t-1, i.e. McmcChain.chain[t] (chain.py:51-54)         */
  int64_t hist_len; /* rows already in every chain's history (len(chain.chain))         */
  int64_t mom_len;  /* rows the running moments (mean, m2) currently cover; equals hist_len
                       for the reference's np.std-over-the-whole-history semantics, smaller
                       after a diagnostics reset.  0 is read as hist_len.              */
  int64_t pending;  /* set by the step entry points.  1 = the LAST of those rows -- every chain's
                       current state X[c], i.e. McmcChain.chain[-1] (chain.py:51-54) -- is counted
                       by hist_len / mom_len but not yet materialised: history row hist_len - 1 is
                       unwritten and mean / m2 lack that sample.  The fused 100-D kernel leaves the
                       row pending because the next generation's proposal stage holds it in registers
                       anyway (no second pass over the moments).  Pass the value back unchanged on the
                       next call; call bpm_flush before reading history / mean / m2.  0 on a new state. */
} bpm_state;

/* RNG-replay buffers for ONE generation: the reference's numpy draws, indexed by
 * GLOBAL chain id (every chain is stepped exactly once per generation, demc.py:103-132).
 * All device pointers.  Per-dimension arrays are dense [n_chains][dim]. */
typedef struct bpm_replay {
  int32_t flip;                /* demc.py:81   flip_bool                                  */
  const int32_t* shuffle_idx;  /* demc.py:84-86 [n_chains]                                */
  const int32_t* cr_idx;       /* dream.py:51  index into CR            (DREAM only)      */
  const double* z;             /* dream.py:52  uniform(0,1,size=dim)    (DREAM only)      */
  const int32_t* fallback_dim; /* dream.py:56  used when the mask is empty (DREAM only)   */
  const int32_t* pairs;        /* [n_chains][del_pairs][2] POOL-LOCAL indices
                                  (demc.py:169, dream.py:66)                              */
  const double* gamma_u;       /* uniform behind the gamma choice (demc.py:175, dream.py:78) */
  const double* e;             /* dream.py:83  var_box values           (DREAM only)      */
  const double* nrm;           /* var_ball values, already scaled (demc.py:182, dream.py:84) */
  const double* accept_u;      /* uniform behind metropolis_accept (samplers.py:336)      */
} bpm_replay;

/* Optional diagnostics written by a generation step; any pointer may be NULL.
 * Indexed by global chain id. */
typedef struct bpm_trace_out {
  int32_t* accept;  /* 1 = proposal accepted */
  double* lnl_prop; /* ln_like(proposal)     */
  double* prop;     /* [n_chains][dim] proposal vectors */
} bpm_trace_out;

/* Batched user likelihood evaluated on the device: theta is [n][ld] (device), write
 * lnl[n] (device), enqueue on `stream`, return 0.  Replaces the scalar
 * ln_like_fn(theta, **kw) frozen at samplers.py:36-43. */
typedef int (*bpm_lnl_fn)(const double* theta, int32_t n, int32_t dim, int32_t ld, double* lnl,
                          void* user, bpm_stream stream);

const char* bpm_last_error(void);
int bpm_version(void);

/* DeMcMpi.__init__ / DreamMpi.__init__ (demc.py:14-32, dream.py:17-30) minus chain
 * storage: creates streams-free workspace for n_chains x dim on cfg->device. */
int bpm_create(const bpm_config* cfg, bpm_handle* out);
int bpm_destroy(bpm_handle h);

/* run_mcmc(**kwargs) re-reads these every call (demc.py:73-75,161-162; dream.py:40-41). */
int bpm_set_run_params(bpm_handle h, double flip, int32_t shuffle, double epsilon,
                       double u_epsilon, double gamma);

/* Select a built-in batched likelihood (replaces the frozen scalar lambda,
 * samplers.py:43).  `params` is a HOST array; layout per target in DESIGN.md. */
int bpm_set_target(bpm_handle h, int32_t target, const double* params, int64_t n_params);
int bpm_set_batched_lnl(bpm_handle h, bpm_lnl_fn fn, void* user);

/* Run-time compiled likelihood (BPM_TARGET_JIT).  `source` is CUDA C++ defining
 *   __device__ double ln_like(const double* theta, const double* data)
 * with theta[BPM_DIM] and data[BPM_NDATA] (both defined as macros; the bpm:: helpers of the
 * library's targets.cuh and the CUDA math functions are in scope).  -inf = outside the prior.
 * The library compiles it with NVRTC for sm_100a together with its own d <= 4 chain-step kernel
 * and a batched row kernel, so the likelihood runs inside the generation kernels.  NVRTC is
 * loaded on first use from $BIPYMC_B200_NVRTC, else the toolkit holding nvcc, else the default
 * loader path.  Compiled cubins are cached for the life of the process (key: translation unit
 * + options); *from_cache (may be NULL) is set to 1 when the cubin came from there.
 * flags: bit 0 = fmad (contract multiply-adds; 0 gives IEEE + - * / rounding of every operation).
 * On a compile error the NVRTC log (line numbers of `source` as "ln_like.cu(line)") goes into
 * log[log_cap].  bpm_jit_compile needs no device.  bpm_set_jit_target compiles (or takes the
 * cached cubin), loads it on the handle's device and copies data[n_data] (HOST) there. */
int bpm_jit_compile(const char* source, int32_t dim, int64_t n_data, int32_t flags, int32_t* from_cache,
                    char* log, int64_t log_cap);
int bpm_set_jit_target(bpm_handle h, const char* source, const double* data, int64_t n_data, int32_t flags,
                       int32_t* from_cache, char* log, int64_t log_cap);

/* Run-time compiled per-observation likelihood (BPM_TARGET_JIT_SUM).  `source` is CUDA C++ defining
 *   __device__ double ln_like_term(const double* theta, const double* row)   -- one observation
 *   __device__ double ln_prior(const double* theta)                          -- only with flags bit 1
 * with theta[BPM_DIM] and row[BPM_ROWLEN]; BPM_NROWS (M) is defined too, and the scope is that of
 * bpm_jit_compile.  data is the row-major [n_rows][row_len] array (HOST), 1 <= n_rows < 2^31.
 *   ln L = ln_prior(theta) + sum over the M rows of ln_like_term(theta, row)
 * (-inf, with no term evaluated, when ln_prior is -inf).  The terms are added in an order fixed by M
 * alone -- chunks of 256 rows, a pairwise tree inside each chunk, an adjacent-pair tree over the chunk
 * partials padded to a power of two, the prior last (bipymc_b200/csrc/kernels_sum.cuh) -- so a given
 * theta gets the same bits whatever the number of chains, the batch size of bpm_eval_lnl, the launch
 * shape or the number of GPUs.  The sum is split over the whole GPU (tiles of chains x groups of
 * chunks); the group partials take at most 2^22 doubles of workspace.  The likelihood runs between
 * the propose and accept kernels at every dim (never in the fused d <= 4 kernel), in serial DE-MC and
 * in bpm_eval_lnl.  flags: bit 0 = fmad, bit 1 = the source defines ln_prior.  Cache, log and
 * from_cache as for bpm_jit_compile; M and row_len are part of the cache key. */
int bpm_jit_compile_sum(const char* source, int32_t dim, int64_t n_rows, int32_t row_len, int32_t flags,
                        int32_t* from_cache, char* log, int64_t log_cap);
int bpm_set_jit_sum_target(bpm_handle h, const char* source, const double* data, int64_t n_rows, int32_t row_len,
                           int32_t flags, int32_t* from_cache, char* log, int64_t log_cap);

/* ln_like for n rows (device in, device out) with the current target. */
int bpm_eval_lnl(bpm_handle h, const double* X, int32_t n, double* lnl, bpm_stream stream);

/* DreamMpi._init_cr / CR state (dream.py:109-117): host arrays of n_cr doubles. */
/* Switch the fused single-kernel fast paths off / on (testing: both must agree). */
int bpm_set_fused(bpm_handle h, int32_t on);

int bpm_set_cr_state(bpm_handle h, const double* p_cr, const double* delta_m,
                     const double* n_cr_updates);
int bpm_get_cr_state(bpm_handle h, double* p_cr, double* delta_m, double* n_cr_updates);

/* Multi-rank CR adaptation (a deliberate change from the reference's per-rank CR
 * state, dream.py:113-117): device pointer to this rank's per-generation partial sums
 * (2*n_cr doubles: jump statistics then counts) for the host's all-reduce, and the
 * p_cr update from the reduced values.  Single-rank handles apply it themselves. */
int bpm_cr_partials(bpm_handle h, double** dev_ptr);
int bpm_apply_cr(bpm_handle h, bpm_stream stream);

/* local_n_accepted / local_n_rejected (demc.py:190,193) and the sticky NaN-alpha flag
 * (numpy raises ValueError("probabilities contain NaN") at samplers.py:336). */
int bpm_get_counters(bpm_handle h, uint64_t* n_accepted, uint64_t* n_rejected, int32_t* nan_alpha);
int bpm_reset_counters(bpm_handle h);

/* DeMcMpi._mcmc_run (demc.py:79-135): n_gen full generations (flip, shuffle, phase a,
 * phase b) with the native Philox stream.  k_gen0 = generation counter of this
 * run_mcmc call (drives the gamma schedule and the burn-in gate); the Philox counter
 * uses st->hist_len so streams never repeat across calls.  st->hist_len is advanced. */
int bpm_step_generations(bpm_handle h, bpm_state* st, int64_t k_gen0, int32_t n_gen,
                         bpm_stream stream);

/* Same generation, but every random draw comes from `rp` (the reference's recorded
 * numpy stream).  Accept decisions must match the reference step for step. */
int bpm_step_generation_replay(bpm_handle h, bpm_state* st, const bpm_replay* rp, int64_t k_gen,
                               const bpm_trace_out* trace, bpm_stream stream);

/* Write the draws the native stream WOULD use for generation (k_gen, st->hist_len)
 * into replay buffers (device, caller-allocated, non-const use of bpm_replay). */
int bpm_dump_draws(bpm_handle h, const bpm_state* st, int64_t k_gen, bpm_replay* out, int32_t* flip,
                   bpm_stream stream);

/* Split generation for likelihoods the library cannot evaluate (scalar Python
 * ln_like_fn, torch callbacks).  Sequence per generation:
 *   bpm_begin_generation; for phase in (0, 1): bpm_propose -> caller fills lnl_prop
 *   -> bpm_accept; bpm_end_generation.
 * prop is [n_phase][ld] in phase order; *n_phase returns the number of chains: all chains of
 * the half on an unsharded handle, only this rank's chains of the half (densely packed, in
 * ascending chain order) on a sharded one (and on d <= 4 handles, which use the packed lists too). */
int bpm_begin_generation(bpm_handle h, bpm_state* st, int64_t k_gen, const bpm_replay* rp_or_null,
                         bpm_stream stream);
int bpm_propose(bpm_handle h, bpm_state* st, int32_t phase, double** prop, int32_t* n_phase,
                bpm_stream stream);
int bpm_accept(bpm_handle h, bpm_state* st, int32_t phase, const double* lnl_prop,
               const bpm_trace_out* trace, bpm_stream stream);
int bpm_end_generation(bpm_handle h, bpm_state* st, bpm_stream stream);
/* One whole half-phase (proposal + built-in / callback likelihood + accept) between
 * bpm_begin_generation and bpm_end_generation: what a multi-rank host calls before
 * its all-gather of the population (demc.py:93,116). */
int bpm_phase(bpm_handle h, bpm_state* st, int32_t phase, bpm_stream stream);

/* Multi-GPU exchange over peer memory.  The reference all-gathers the whole population
 * before each half-phase (comm.Allgather, demc.py:93,116).  Here every rank keeps a replica
 * of X; with peers set, the accept stage of every kernel stores an ACCEPTED chain's new row
 * into each peer replica as well (NVLink peer stores from inside the kernel), so only the
 * rows that changed cross the fabric and no separate gather runs.  The host still has to
 * put a cross-rank barrier between half-phases (any tiny collective on the same stream).
 *   bpm_dev_alloc / bpm_dev_free : plain cudaMalloc'ed memory (IPC-exportable) for X
 *   bpm_ipc_export : 64-byte cudaIpcMemHandle of such an allocation (send it to the peers)
 *   bpm_ipc_open / bpm_ipc_close : map a peer's allocation into this process
 *   bpm_set_peers : device pointers (mapped here) of the OTHER ranks' X replicas, same
 *                   [n_chains][ld] layout; n_peers = 0 switches the peer stores off.     */
int bpm_dev_alloc(int32_t device, uint64_t bytes, void** dev_ptr);
int bpm_dev_free(int32_t device, void* dev_ptr);
int bpm_ipc_export(int32_t device, const void* dev_ptr, unsigned char handle64[64]);
int bpm_ipc_open(int32_t device, const unsigned char handle64[64], void** dev_ptr);
int bpm_ipc_close(int32_t device, void* dev_ptr);
int bpm_set_peers(bpm_handle h, double* const* peer_X, int32_t n_peers);
/* Plain asynchronous copy between two device pointers of this process' address space, either of which may
 * be a peer allocation mapped with bpm_ipc_open (NVLink copy engines): the sub-population re-deal pulls its
 * chains out of the other islands with it (NCCL's all-to-all moved the same 30 GB per rank at ~20 GB/s). */
int bpm_peer_copy(int32_t device, void* dst, const void* src, uint64_t bytes, bpm_stream stream);

/* Peer-memory barrier: the comm.Barrier() of demc.py:135 and the synchronisation implied by the two
 * Allgathers (demc.py:93,116) without a collective library on the path.  Every rank allocates one sync
 * block of bpm_sync_bytes() zeroed bytes with bpm_dev_alloc, exchanges its IPC handle, maps the others
 * and registers all of them, indexed by rank (blocks[rank] = its own).  With a sync set,
 * bpm_step_generations works on SHARDED handles: it puts a barrier kernel (a few microseconds on the
 * same stream) after each half-phase and folds the all-reduce of the 2 n_cr CR statistics into the one
 * that closes a DREAM generation (sums added in rank order: identical bits on every rank).  All ranks
 * must make the same sequence of calls.  bpm_peer_barrier: one barrier on `stream` (e.g. after the host
 * refreshed the replicas by other means).  A peer that does not arrive within ~4 s raises a sticky flag
 * instead of hanging the device: bpm_sync_error.  world = 0 switches the sync off. */
int bpm_sync_bytes(uint64_t* bytes);
int bpm_set_sync(bpm_handle h, void* const* blocks, int32_t rank, int32_t world);
int bpm_peer_barrier(bpm_handle h, bpm_stream stream);
int bpm_sync_error(bpm_handle h, int32_t* err);

/* Host-buffer entry (the end-to-end path): X_host / lnl_host are HOST arrays (pinned
 * for full speed); copies them to the device, runs n_gen native generations, copies the
 * result back.  Synchronous.  The chain HISTORY stays with the caller (the host arrays are
 * McmcChain.current_pos of every chain; appending them is the caller's np.vstack, chain.py:51-54).
 * What DREAM derives from the history -- the per-chain running mean / M2 behind np.std(chain.chain)
 * (dream.py:128) -- is kept on the device by the handle between calls, so crossover adaptation runs
 * exactly as in bpm_step_generations: the moments start with the population of the first call
 * (g_abs0 = the chains' length then) and see every population handed in afterwards.
 * bpm_host_entry_restart forgets them (a new sampling run through the same handle). */
int bpm_generations_host(bpm_handle h, double* X_host, double* lnl_host, int64_t k_gen0,
                         int64_t g_abs0, int32_t n_gen);
int bpm_host_entry_restart(bpm_handle h);
/* The same end-to-end step for a SHARDED population (one process per GPU; needs bpm_set_peers and
 * bpm_set_sync).  X_host [n_local][ld] / lnl_host [n_local] are THIS rank's chains in pinned
 * (device-mapped) host memory; st is the rank's device state (st->X = its full replica).  One kernel reads
 * the shard over PCIe (zero-copy) and stores every piece into the rank's own and all peer replicas
 * (host->device copy and the reference's Allgather, demc.py:93, fused; BIPYMC_B200_SHARD_DMA=1 selects the
 * copy-engine form: chunked host copies, each chunk forwarded by peer copies), a peer barrier follows,
 * n_gen generations run with the host array registered as one more replica -- so accepted rows are
 * written back by the phase kernels themselves -- and the cached likelihoods come back with one copy.
 * Collective: every rank calls it with the same k_gen0 / n_gen.  Synchronous. */
int bpm_generations_host_sharded(bpm_handle h, bpm_state* st, double* X_host, double* lnl_host,
                                 int64_t k_gen0, int32_t n_gen, bpm_stream stream);
/* When both host arrays are pinned (device-mapped) memory, bpm_generations_host writes back only
 * the rows of chains that moved (the device stores them straight into the host arrays; rows of
 * chains that did not move are already correct there).  Bytes the last call moved device->host. */
int bpm_last_d2h_bytes(bpm_handle h, uint64_t* bytes);

/* Materialise a pending row (bpm_state.pending): writes history row hist_len - 1 from X and folds it
 * into mean / m2 with the kernels' own Welford arithmetic, then clears st->pending.  No-op when nothing
 * is pending.  st->history must be the base the step call that left the row pending was given.
 * Every entry point that needs the row (replay steps, the eager kernels, diagnostics) calls it itself;
 * the host calls it before READING history / mean / m2 (McmcChain.chain, param_est, save_state). */
int bpm_flush(bpm_handle h, bpm_state* st, bpm_stream stream);

/* Rebuild running moments from a stored history (load_state / warm start). */
int bpm_moments_from_history(bpm_handle h, bpm_state* st, bpm_stream stream);

/* Additions the north star asks for (not in the reference; Vrugt et al. 2009, the paper
 * cited at readme.md:41-43).
 *
 * IQR outlier-chain reset.  Omega_c = mean log-density of chain c over a trailing window.
 * bpm_omega_track(h, 1) zeroes and starts a per-chain running sum of the cached ln_like,
 * advanced once per generation by the step entry points; bpm_omega returns the device
 * array of sums (global chain index; only local rows are maintained) and the number of
 * generations summed.  bpm_outlier_reset: chains with Omega_c < Q1 - 2 (Q3 - Q1)
 * (numpy.percentile's linear rule over ALL n_chains) take the state, cached ln_like and
 * Omega sum of the best chain (argmax Omega, lowest id on ties).  `omega` = device
 * [n_chains] means for every chain (a sharded host all-gathers them, and st->lnl / st->X
 * must then be current for all chains), or NULL to use the tracked sums of an unsharded
 * handle.  Only local chains are written.  Optional outputs: flags_dev [n_chains] device
 * (1 = reset, local rows only), *n_reset host count, stats_host[4] = {threshold, Q1, Q3,
 * best chain}; asking for a host output synchronises the stream. */
int bpm_omega_track(bpm_handle h, int32_t on);
int bpm_omega(bpm_handle h, double** sum_dev, int64_t* count);
int bpm_outlier_reset(bpm_handle h, bpm_state* st, const double* omega, int32_t* flags_dev,
                      int32_t* n_reset, double* stats_host, bpm_stream stream);
/* Streaming posterior covariance (north_star: "posterior mean and covariance ... within Monte-Carlo
 * standard error"; the reference gets it from the stored super chain, demc.py:235-248).  While on, every
 * generation adds this rank's chain states to sum[d] and cross[d][d] (= sum x x^T) on the device;
 * O(n_local d^2) per generation, meant for diagnostic runs.  bpm_cov_track(h, 1) zeroes and starts,
 * (h, 0) stops; bpm_cov_read copies the sums and the number of generations accumulated to the host
 * (covariance = cross / n - mean mean^T with n = generations * n_local; a sharded host adds the ranks'
 * sums first).  Synchronises the device. */
int bpm_cov_track(bpm_handle h, int32_t on);
int bpm_cov_read(bpm_handle h, double* sum_host, double* cross_host, int64_t* generations);

/* Gelman-Rubin R-hat per dimension over this handle's local chains: from history rows
 * [t0, hist_len) when t0 >= 0, from the running moments (mean, m2 over mom_len rows) when
 * t0 < 0.  rhat_host: dim doubles.  Synchronises the stream. */
int bpm_rhat(bpm_handle h, const bpm_state* st, int64_t t0, double* rhat_host, bpm_stream stream);

/* Per-kernel timing for the benchmark's roofline line: while on, every launch is
 * bracketed by CUDA events on the caller's stream.  bpm_profile_read synchronises and
 * returns total milliseconds and launch counts for 8 kinds: 0 split/shuffle, 1 propose,
 * 2 likelihood, 3 accept, 4 fused half-phase, 5 CR reduction, 6 peer barrier / CR exchange, 7 host shard
 * copy-in + all-gather; then clears the records. */
int bpm_profile(bpm_handle h, int32_t on);
int bpm_profile_read(bpm_handle h, double* ms_by_kind8, int64_t* launches_by_kind8);

/* Host-side mirrors of the device RNG (the same source compiled for the host) so a
 * CPU-only test-suite can check known-answer vectors and the shuffle permutation. */
int bpm_test_philox(const uint32_t* ctr4, const uint32_t* key2, uint32_t* out4);
int bpm_test_permutation(uint64_t seed, uint64_t g_abs, int32_t n, int32_t* out_perm);

#ifdef __cplusplus
}
#endif
#endif /* BIPYMC_B200_H_ */
