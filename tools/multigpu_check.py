#!/usr/bin/env python
"""Launched under torchrun with G >= 2 ranks (one per GPU, NCCL): a sharded DREAM / DE-MC run
must reproduce the single-GPU run of the same seed.  With CR adaptation off the chains are
bit-identical (every draw is a function of (seed, generation, chain), never of the rank);
with adaptation on p_cr agrees to rounding of the all-reduced sums.  Rank 0 prints
MULTIGPU_OK on success."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LINEFIT_CUDA = r'''
__device__ double ln_like(const double* theta, const double* data) {
  const int M = BPM_NDATA / 3;
  return bpm::linefit_lnl(data, data + M, data + 2 * M, M, theta[0], theta[1], theta[2]);
}
'''
LINEFIT_TERM = r'''
__device__ double ln_like_term(const double* theta, const double* row) {
  const double model = theta[0] * row[0] + theta[1];
  const double inv = 1.0 / (row[2] * row[2] + model * model * exp(2.0 * theta[2]));
  const double r = row[1] - model;
  return -0.5 * (r * r * inv - log(inv));
}
'''


def main():
    rank = int(os.environ["RANK"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    from bipymc_b200 import DreamMpi, DeMcMpi, targets
    from bipymc_b200.demc import _SingleComm
    world = dist.get_world_size()
    lf = targets.LineFit()
    cases = [
        ("dream-gauss100", DreamMpi, targets.Gauss_100D(), np.zeros(100), 4096 + 2 * world, dict(burnin_gen=0), 1.0),
        ("dream-gauss100-adapt", DreamMpi, targets.Gauss_100D(), np.zeros(100), 2048, dict(burnin_gen=1000, n_cr_gen=2), 1.0),
        ("demc-banana", DeMcMpi, targets.Banana_2D(), [0.0, 0.0], 1000 * world, {}, 0.5),
        # d > 112: generic split path with the FP64 tensor-pipe likelihood and device-counted row lists
        ("dream-gauss128", DreamMpi, targets.Gauss_100D(dim=128), np.zeros(128), 640 + 2 * world, dict(burnin_gen=0), 1.0),
        ("dream-linefit-outlier", DreamMpi, targets.LineFit(), [-0.8, 4.5, 0.2], 512 * world,
         dict(burnin_gen=1000, n_cr_gen=3, outlier_gen=5), 1e-2),
        # user likelihood compiled at run time (BPM_TARGET_JIT): the fused d <= 4 kernel with in-kernel peer stores
        ("dream-linefit-cuda", DreamMpi, lf, [-0.8, 4.5, 0.2], 512 * world,
         dict(burnin_gen=0, ln_like_cuda=targets.CudaLikelihood(LINEFIT_CUDA, 3, np.concatenate([lf.x, lf.y, lf.yerr]))),
         1e-2),
        # per-observation source summed across the GPU (BPM_TARGET_JIT_SUM): the split path with device-counted lists
        ("dream-linefit-cuda-sum", DreamMpi, lf, [-0.8, 4.5, 0.2], 512 * world,
         dict(burnin_gen=0, ln_like_cuda=targets.CudaSumLikelihood(LINEFIT_TERM, 3, np.stack([lf.x, lf.y, lf.yerr], 1))),
         1e-2),
    ]
    G = 12
    runs = [(c, ex) for c in cases for ex in ("p2p", "allgather")]
    for (name, cls, tgt, th0, N, kw, veps), exchange in runs:
        np.random.seed(3)
        s = cls(tgt.ln_like, th0, n_chains=N, seed=5, varepsilon=veps, device=local, exchange=exchange, **kw)
        assert s.comm.size == world
        if exchange == "p2p" and s._exchange != "p2p" and rank == 0:
            print("NOTE: no peer access on this box, p2p fell back to", s._exchange, flush=True)
        s.run_mcmc(N * (G + 1))
        full = s.super_chain_mpi(0)
        acc = (s.n_accepted, s.n_rejected)
        rh = s.rhat()
        if rank == 0:
            np.random.seed(3)
            one = cls(tgt.ln_like, th0, n_chains=N, seed=5, varepsilon=veps, device=local,
                      mpi_comm=_SingleComm(), **kw)
            one.run_mcmc(N * (G + 1))
            ref = one.super_chain
            assert full.shape == ref.shape, (full.shape, ref.shape)
            exact = "adapt" not in name and "outlier" not in name
            if exact:
                assert np.array_equal(full, ref), "%s: sharded run differs from the single-GPU run" % name
                assert acc == (one.n_accepted, one.n_rejected + world - 1), (acc, one.n_accepted, one.n_rejected)
            else:
                # all-reduced CR sums round differently from the single-rank block order
                frac = np.mean(np.all(full == ref, axis=1))
                assert frac > 0.9, "%s: only %.3f of rows identical" % (name, frac)
                np.testing.assert_allclose(s.p_cr, one.p_cr, rtol=1e-6)
            np.testing.assert_allclose(rh, one.rhat(), rtol=1e-6 if not exact else 1e-9)
            if "outlier" in name:
                print(name, "resets", s.n_outlier_resets, one.n_outlier_resets)
            print("case", name, exchange, "->", s._exchange, "ok", flush=True)
        dist.barrier()
        del s
    # ---- serial DeMc (delayed accept) on several ranks: every chain of a sweep reads ALL other chains of the frozen
    #      population, so the ranks exchange with an all-gather after the sweep, never with in-kernel peer stores
    #      (ADVICE r1); the sharded sweep must reproduce the single-GPU one bit for bit
    from bipymc_b200 import DeMc
    Ns = 64 * world
    np.random.seed(4)
    sd = DeMc(targets.Banana_2D().ln_like, n_chains=Ns, seed=6, device=local, exchange="p2p")
    assert sd._exchange == "allgather"
    sd.run_mcmc(Ns * 9, [0.0, 0.0], varepsilon=1e-2)
    full = sd.super_chain_mpi(0)
    if rank == 0:
        np.random.seed(4)
        one = DeMc(targets.Banana_2D().ln_like, n_chains=Ns, seed=6, device=local, mpi_comm=_SingleComm())
        one.run_mcmc(Ns * 9, [0.0, 0.0], varepsilon=1e-2)
        assert np.array_equal(full, one.super_chain), "sharded serial sweep differs from the single-GPU sweep"
        print("case serial-demc sharded ok", flush=True)
    dist.barrier()
    del sd
    # ---- sharded end-to-end entry (bpm_generations_host_sharded): host shards in / out every generation ==
    #      the device-resident sharded run of the same seed (adaptation on: moments live in the sampler state)
    import ctypes as C
    from bipymc_b200 import _lib
    N, d, G = 2048 * world, 100, 6
    tgt = targets.Gauss_100D()
    kw = dict(n_chains=N, seed=5, varepsilon=1.0, device=local, history="none", burnin_gen=1000, n_cr_gen=2)
    np.random.seed(3)
    ref = DreamMpi(tgt.ln_like, np.zeros(d), **kw)
    ref.run_mcmc(N * (G + 1))
    np.random.seed(3)
    s = DreamMpi(tgt.ln_like, np.zeros(d), **kw)
    assert s._sync_on, "peer-memory barrier not available"
    s.run_mcmc(N)                                   # run parameters + initial likelihoods, no generation
    lo, hi = int(s.rank_chain_ids[0]), int(s.rank_chain_ids[-1]) + 1
    Xh = torch.empty((hi - lo, s._ld), dtype=torch.float64).pin_memory()
    Lh = torch.empty((hi - lo,), dtype=torch.float64).pin_memory()
    Xh.copy_(s._X[lo:hi]); Lh.copy_(s._lnl[lo:hi])
    st = s._state(None)
    for g in range(G):
        _lib.check(s._libh.bpm_generations_host_sharded(s._handle, C.byref(st), Xh.data_ptr(), Lh.data_ptr(), g, 1,
                                                        s._stream()))
    torch.cuda.synchronize()
    assert torch.equal(Xh, ref._X[lo:hi].cpu()), "host shard differs from the device-resident sharded run"
    assert torch.equal(Lh, ref._lnl[lo:hi].cpu())
    assert torch.equal(s._X, ref._X), "replicas (all shards) differ"
    assert np.array_equal(s.p_cr, ref.p_cr)
    dist.barrier()
    if rank == 0:
        print("case host-sharded entry ok", flush=True)
    s.close(); ref.close()
    # ---- sub-population (island) mode: no replica, chains re-dealt every k generations
    N, k = 1024 * world, 5
    np.random.seed(3)
    s = DreamMpi(targets.Banana_2D().ln_like, [0.0, 0.0], n_chains=N, seed=5, varepsilon=0.5, device=local,
                 subpop_k=k, burnin_gen=1000, n_cr_gen=3)
    nl = len(s.rank_chain_ids)
    assert s._X.shape[0] == nl and s._lnl.shape[0] == nl, "an island holds only its own chains"
    # the re-deal is a permutation of the chains: tag every chain with its global id and deal once
    keepX, keepM = s._X.clone(), s._mean.clone()
    s._X[:, 0] = torch.arange(int(s.rank_chain_ids[0]), int(s.rank_chain_ids[-1]) + 1, device=dev, dtype=torch.float64)
    s._mean.copy_(s._X)
    s._redeal()
    tags = s._X[:, 0].round().long()
    assert torch.equal(s._mean[:, 0].round().long(), tags), "moments travel with their chain"
    origin = torch.div(tags, nl, rounding_mode="floor")
    per_origin = torch.bincount(origin, minlength=world)
    assert int(per_origin.min()) == int(per_origin.max()) == nl // world, per_origin
    allt = [torch.empty_like(tags) for _ in range(world)]
    dist.all_gather(allt, tags)
    assert torch.equal(torch.sort(torch.cat(allt))[0], torch.arange(N, device=dev)), "no chain lost or duplicated"
    # undo (world deals of this pattern are not the identity in general: just restore)
    s._X.copy_(keepX); s._mean.copy_(keepM); s._gens_since_deal = 0
    G = 23
    s.run_mcmc(N * (G + 1))
    assert s.n_accepted + s.n_rejected == N * G + world, (s.n_accepted, s.n_rejected)
    assert s._gens_since_deal == G and s.am_chains[0].chain_len == G + 1
    rh = s.rhat()
    m, sd = s.moment_estimates()
    sc = s.super_chain_mpi(0)
    if rank == 0:
        assert sc.shape == (N * (G + 1), 2) and np.all(np.isfinite(sc)) and np.all(np.isfinite(rh))
        assert abs(m[0]) < 0.5 and 0.2 < sd[0] < 3.0, (m, sd)
        print("case subpop k=%d ok" % k, "rhat", rh, flush=True)
    dist.barrier()
    if rank == 0:
        print("MULTIGPU_OK", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
