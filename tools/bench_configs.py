#!/usr/bin/env python
"""Secondary measurements for the BASELINE configs that are NOT the headline bench line
(bench.py measures configs[1]).  Prints one JSON line per configuration:
  c3  DREAM, bimodal 2-D Gaussian, 10^6 chains, CR adaptation + outlier reset on, no history
  c4  DREAM, line fit (3 parameters, 50 data points), 10^5 chains
  c4_cuda_same / c4_cuda / c4_torch  the same run with the likelihood as a run-time compiled CUDA
      source calling the built-in's bpm::linefit_lnl / in the reference's per-term form (fmad=False) /
      as examples/ex_para_fit_b200.py's batched torch function
  expfit / expfit_cuda / expfit_torch  DREAM on the 5-parameter exp fit (60 points), 10^5 chains:
      built-in split path / the reference's form as CUDA source (fmad=False) / torch ops
  expfit_sum_N<N>_M<M> / expfit_cuda_N<N>_M<M>  the exp fit on targets.expfit_data(n=M) with N chains, as a
      per-observation CudaSumLikelihood / as a whole-function CudaLikelihood (both fmad=False, the reference's
      arithmetic): N1024_M1e5, N1e5_M1e4, N1024_M1e6 (sum only)
  c4_sum  c4 with the reference's per-term line fit as a CudaSumLikelihood (fmad=False), against c4_cuda
  demc100  DE-MC on the 100-D Gaussian, 10^5 chains (32 d + 16 bytes per chain-step)
Device-resident timing with CUDA events, same rules as bench.py."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402


def run(name, make, N, d, bytes_per_step, gens=100, warm=20, extra=None, terms_per_gen=None):
    from bipymc_b200 import _lib
    np.random.seed(1)
    s = make()
    k = 0
    s.run_mcmc(N * (warm + 1))
    k += warm
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    s.run_mcmc(N * (gens + 1), _k_gen0=k)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    v = N * gens / (ms * 1e-3)
    peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if os.path.exists(
        os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
    # untimed extra pass with CUDA events around every launch: average launch time per kernel family
    import ctypes as C
    pg = max(4, gens // 5)
    _lib.check(s._libh.bpm_profile(s._handle, 1))
    s.run_mcmc(N * (pg + 1), _k_gen0=k + gens)
    torch.cuda.synchronize()
    ms_k, n_k = (C.c_double * 8)(), (C.c_int64 * 8)()
    _lib.check(s._libh.bpm_profile_read(s._handle, ms_k, n_k))
    _lib.check(s._libh.bpm_profile(s._handle, 0))
    kinds = ["split", "propose", "likelihood", "accept", "fused_phase", "cr_reduce", "other6", "other7"]
    kms = dict((kinds[i], {"avg_ms": ms_k[i] / n_k[i], "per_generation": n_k[i] / pg}) for i in range(8) if n_k[i])
    if terms_per_gen:       # likelihood terms (chains x observations) per generation over likelihood time per generation
        extra = dict(extra or {}, terms_per_s=terms_per_gen / (ms_k[2] / pg * 1e-3), likelihood_avg_ms=ms_k[2] / n_k[2])
    print(json.dumps(dict({"config": name, "n_chains": N, "dim": d, "chain_steps_per_s": v, "ms_per_generation": ms / gens,
                      "algorithmic_bytes_per_chain_step": bytes_per_step,
                      "algorithmic_GBps": v * bytes_per_step / 1e9, "frac_of_hbm_peak": v * bytes_per_step / 1e9 / peak,
                      "acceptance_fraction": s.acceptance_fraction, "launches_event_pass": kms}, **(extra or {}))))
    s.close()


LINEFIT_SAME = r'''
__device__ double ln_like(const double* theta, const double* data) {
  const int M = BPM_NDATA / 3;
  return bpm::linefit_lnl(data, data + M, data + 2 * M, M, theta[0], theta[1], theta[2]);
}
'''

# ex_exp_fit.py:73-121 as written there (one data point at a time); data = t[M], y[M]
EXPFIT_CUDA = r'''
__device__ double ln_like(const double* th, const double* data) {
  const int M = BPM_NDATA / 2;
  const double tau = th[0], c_inf = th[1], c_0 = th[2], leak = th[3], sigma = th[4];
  if (!(-5.0 < c_inf && c_inf < 5.0 && 1.0 < tau && tau < 50.0 && -1.0 < c_0 && c_0 < 1.0 &&
        -5.0 < leak && leak < 5.0 && 0.0 < sigma && sigma < 1.0)) return -INFINITY;
  double s = 0.0;
  for (int i = 0; i < M; ++i) {
    const double t = data[i];
    const double m = c_inf + c_0 * -1.0 * exp(-t / tau) - leak * t;
    s += (m - data[M + i]) * (m - data[M + i]) / sigma - log(1.0 / sigma);
  }
  return 0.0 + -0.5 * s;
}
'''


# the same two models per observation (targets.CudaSumLikelihood); rows = (t, y) / (x, y, yerr)
EXPFIT_TERM = r'''
__device__ double ln_like_term(const double* th, const double* row) {
  const double m = th[1] + th[2] * -1.0 * exp(-row[0] / th[0]) - th[3] * row[0];
  return -0.5 * ((m - row[1]) * (m - row[1]) / th[4] - log(1.0 / th[4]));
}
'''
EXPFIT_PRIOR = r'''
__device__ double ln_prior(const double* th) {
  const double tau = th[0], c_inf = th[1], c_0 = th[2], leak = th[3], sigma = th[4];
  return (-5.0 < c_inf && c_inf < 5.0 && 1.0 < tau && tau < 50.0 && -1.0 < c_0 && c_0 < 1.0 &&
          -5.0 < leak && leak < 5.0 && 0.0 < sigma && sigma < 1.0) ? 0.0 : -INFINITY;
}
'''
LINEFIT_TERM = r'''
__device__ double ln_like_term(const double* theta, const double* row) {
  const double model = theta[0] * row[0] + theta[1];
  const double inv = 1.0 / (row[2] * row[2] + model * model * exp(2.0 * theta[2]));
  return -0.5 * ((row[1] - model) * (row[1] - model) * inv - log(inv));
}
'''
LINEFIT_PRIOR = r'''
__device__ double ln_prior(const double* theta) {
  const double m = theta[0], b = theta[1], lnf = theta[2];
  return (-5.0 < m && m < 0.5 && 0.0 < b && b < 10.0 && -10.0 < lnf && lnf < 1.0) ? 0.0 : -INFINITY;
}
'''


def _expfit_torch(t, y):
    def lnprob(th):
        tau, c_inf, c_0, leak, sigma = (th[:, i:i + 1] for i in range(5))
        m = c_inf + c_0 * -1.0 * torch.exp(-t[None, :] / tau) - leak * t[None, :]
        ll = 0.0 + -0.5 * ((m - y[None, :]) ** 2 / sigma - torch.log(1.0 / sigma)).sum(dim=1)
        ok = (th[:, 1] > -5) & (th[:, 1] < 5) & (th[:, 0] > 1) & (th[:, 0] < 50) & (th[:, 2] > -1) & (th[:, 2] < 1) & \
             (th[:, 3] > -5) & (th[:, 3] < 5) & (th[:, 4] > 0) & (th[:, 4] < 1)
        return torch.where(ok, ll, torch.full_like(ll, -float("inf")))
    return lnprob


def _plain(target):
    """The target's scalar ln_like hidden behind a lambda: a built-in target's own method would select the
    built-in device likelihood, which takes precedence over ln_like_batched."""
    return lambda theta: target.ln_like(theta)


def _nvrtc_loaded():
    """Path (symlinks resolved: the file name carries the version) of the NVRTC this process loaded."""
    with open("/proc/self/maps") as f:
        for line in f:
            if "libnvrtc.so" in line:
                return os.path.realpath(line.split()[-1])
    return None


def _cuda_lik(src, dim, data, fmad, cls=None, **kw):
    """CudaLikelihood (or cls) plus its compile time: first compile of the source in this process, then the cached
    one."""
    import time
    from bipymc_b200 import targets
    lik = (cls or targets.CudaLikelihood)(src, dim, data, fmad=fmad, **kw)
    t0 = time.perf_counter()
    first_cached = lik.compile()
    t1 = time.perf_counter()
    assert lik.compile()
    t2 = time.perf_counter()
    return lik, {"compile_s": t1 - t0, "compile_was_cached": first_cached, "compile_cached_s": t2 - t1,
                 "nvrtc": _nvrtc_loaded()}


def main():
    from bipymc_b200 import DreamMpi, DeMcMpi, targets
    which = sys.argv[1:] or ["c3", "c4", "demc100", "c5shape"]
    c4_kw = dict(n_chains=100000, seed=3, varepsilon=1e-2, history="none", burnin_gen=10 ** 6, n_cr_gen=10)
    c4_bytes = 64 * 3 + 16 + 32 * 3 + 8 * 3
    ex_kw = dict(n_chains=100000, seed=3, varepsilon=np.asarray([1e-2, 1e-2, 1e-3, 1e-8, 1e-9]) * 1e-2,
                 history="none", burnin_gen=10 ** 6, n_cr_gen=10)                   # ex_exp_fit.py:135
    ex_bytes = 64 * 5 + 16 + 32 * 5 + 8 * 5
    ex_th0 = [12.0, 1.5, 0.6, 1e-3, 2e-3]
    lf, ef = targets.LineFit(), targets.ExpFit()
    lf_data, ef_data = np.concatenate([lf.x, lf.y, lf.yerr]), np.concatenate([ef.t, ef.y])
    if "c3" in which:
        N = 1000000
        t = targets.BimodeGauss_2D(log_of_pdf=False)
        # own row + 6 partners + write (8 d each) + lnL r/w, + moments r/w (32 d) during adaptation
        run("c3 bimodal DREAM 1e6 chains", lambda: DreamMpi(t.ln_like, [0.0, 0.0], n_chains=N, seed=3, varepsilon=1.0,
                                                              history="none", burnin_gen=10 ** 6, n_cr_gen=10,
                                                              outlier_gen=50), N, 2, 64 * 2 + 16 + 32 * 2 + 8 * 2)
    if "c4" in which:
        N = 100000
        t = targets.LineFit()
        run("c4 linefit DREAM 1e5 chains", lambda: DreamMpi(t.ln_like, [-0.8, 4.5, 0.2], n_chains=N, seed=3,
                                                              varepsilon=1e-2, history="none", burnin_gen=10 ** 6,
                                                              n_cr_gen=10), N, 3, 64 * 3 + 16 + 32 * 3 + 8 * 3)
    if "c4_cuda_same" in which:
        lik, info = _cuda_lik(LINEFIT_SAME, 3, lf_data, True)
        run("c4_cuda_same linefit (bpm::linefit_lnl as CUDA source) DREAM 1e5 chains",
            lambda: DreamMpi(lf.ln_like, [-0.8, 4.5, 0.2], ln_like_cuda=lik, **c4_kw), 100000, 3, c4_bytes, extra=info)
    if "c4_cuda" in which:
        sys.path.insert(0, os.path.join(ROOT, "examples"))
        from ex_para_fit_b200 import LNPROB_CUDA
        lik, info = _cuda_lik(LNPROB_CUDA, 3, lf_data, False)
        run("c4_cuda linefit (reference per-term form as CUDA source, fmad=False) DREAM 1e5 chains",
            lambda: DreamMpi(lf.ln_like, [-0.8, 4.5, 0.2], ln_like_cuda=lik, **c4_kw), 100000, 3, c4_bytes, extra=info)
    if "c4_torch" in which:
        sys.path.insert(0, os.path.join(ROOT, "examples"))
        from ex_para_fit_b200 import make_lnprob_batched
        fb = make_lnprob_batched(*(torch.from_numpy(v).cuda() for v in (lf.x, lf.y, lf.yerr)))
        assert DreamMpi(_plain(lf), [-0.8, 4.5, 0.2], ln_like_batched=fb, n_chains=8)._mode() == "batched"
        run("c4_torch linefit (batched torch plug-in) DREAM 1e5 chains",
            lambda: DreamMpi(_plain(lf), [-0.8, 4.5, 0.2], ln_like_batched=fb, **c4_kw), 100000, 3, c4_bytes,
            gens=50, warm=10)
    if "expfit" in which:
        run("expfit DREAM d=5 1e5 chains (built-in)", lambda: DreamMpi(ef.ln_like, ex_th0, **ex_kw), 100000, 5, ex_bytes)
    if "expfit_cuda" in which:
        lik, info = _cuda_lik(EXPFIT_CUDA, 5, ef_data, False)
        run("expfit_cuda DREAM d=5 1e5 chains (reference form as CUDA source, fmad=False)",
            lambda: DreamMpi(ef.ln_like, ex_th0, ln_like_cuda=lik, **ex_kw), 100000, 5, ex_bytes, extra=info)
    if "expfit_torch" in which:
        fe = _expfit_torch(*(torch.from_numpy(v).cuda() for v in (ef.t, ef.y)))
        run("expfit_torch DREAM d=5 1e5 chains (batched torch plug-in)",
            lambda: DreamMpi(_plain(ef), ex_th0, ln_like_batched=fe, **ex_kw), 100000, 5, ex_bytes, gens=50, warm=10)
    sum_runs = {"expfit_sum_N1024_M1e5": (1024, 100000), "expfit_cuda_N1024_M1e5": (1024, 100000),
                "expfit_sum_N1e5_M1e4": (100000, 10000), "expfit_cuda_N1e5_M1e4": (100000, 10000),
                "expfit_sum_N1024_M1e6": (1024, 1000000)}
    for name in [w for w in which if w in sum_runs]:
        N, M = sum_runs[name]
        t, y = targets.expfit_data(n=M)
        if "_sum_" in name:
            lik, info = _cuda_lik(EXPFIT_TERM + EXPFIT_PRIOR, 5, np.stack([t, y], 1), False, targets.CudaSumLikelihood,
                                  prior=True)
        else:
            lik, info = _cuda_lik(EXPFIT_CUDA, 5, np.concatenate([t, y]), False)
        slow = N * M >= 10 ** 9
        run(name + " DREAM d=5 exp fit", lambda: DreamMpi(ef.ln_like, ex_th0, ln_like_cuda=lik, **dict(ex_kw, n_chains=N)),
            N, 5, ex_bytes, gens=10 if slow else 50, warm=3 if slow else 10, extra=dict(info, n_obs=M),
            terms_per_gen=N * M)
    if "c4_sum" in which:
        lik, info = _cuda_lik(LINEFIT_TERM + LINEFIT_PRIOR, 3, np.stack([lf.x, lf.y, lf.yerr], 1), False,
                              targets.CudaSumLikelihood, prior=True)
        run("c4_sum linefit (reference per-term form as CudaSumLikelihood, fmad=False) DREAM 1e5 chains",
            lambda: DreamMpi(lf.ln_like, [-0.8, 4.5, 0.2], ln_like_cuda=lik, **c4_kw), 100000, 3, c4_bytes,
            extra=dict(info, n_obs=lf.x.size), terms_per_gen=100000 * lf.x.size)
    if "demc100" in which:
        N = 100000
        t = targets.Gauss_100D()
        run("DE-MC Gauss_100D 1e5 chains", lambda: DeMcMpi(t.ln_like, np.zeros(100), n_chains=N, seed=3,
                                                             varepsilon=np.arange(100) + 1.0, history="none"),
            N, 100, 32 * 100 + 16 + 32 * 100)


def c5shape():
    """configs[4] shape on one GPU: DREAM on the 1000-D correlated Gaussian (direct log-density),
    2 x 10^4 chains -- the generic split path (propose / tiled FP64 quadratic form / accept)."""
    from bipymc_b200 import DreamMpi, targets
    N, d = 20000, 1000
    t = targets.Gauss_100D(dim=d)
    run("c5-shape DREAM Gauss_1000D 2e4 chains", lambda: DreamMpi(t.ln_like, np.zeros(d), n_chains=N, seed=3,
                                                                    varepsilon=np.arange(d) + 1.0, history="none",
                                                                    burnin_gen=10 ** 6, n_cr_gen=10),
        N, d, 64 * d + 16 + 32 * d + 8 * d, gens=20, warm=12)


def c5multi():
    """configs[4] shape sharded over the GPUs of one box (launch under torchrun): DREAM on the
    1000-D Gaussian, 2.5 x 10^4 chains per GPU, once as ONE population (replicas + peer-memory
    exchange) and once in the stated sub-population mode (islands re-dealt every 10 generations)."""
    import torch.distributed as dist
    from bipymc_b200 import DreamMpi, targets
    rank, local = int(os.environ["RANK"]), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    world = dist.get_world_size()
    N, d, gens, warm = 25000 * world, 1000, 20, 10
    t = targets.Gauss_100D(dim=d)
    for mode, kw in (("one population, p2p exchange", {}), ("sub-population mode k=10", dict(subpop_k=10))):
        np.random.seed(1)
        s = DreamMpi(t.ln_like, np.zeros(d), n_chains=N, seed=3, varepsilon=np.arange(d) + 1.0, history="none",
                     burnin_gen=10 ** 6, n_cr_gen=5, device=local, **kw)
        s.run_mcmc(N * (warm + 1))
        torch.cuda.synchronize(); dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        s.run_mcmc(N * (gens + 1), _k_gen0=warm)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if rank == 0:
            print(json.dumps({"config": "c5-shape DREAM Gauss_1000D, %d GPUs x 2.5e4 chains, %s" % (world, mode),
                              "n_chains": N, "chain_steps_per_s": N * gens / (float(ms.item()) * 1e-3),
                              "ms_per_generation": float(ms.item()) / gens,
                              "acceptance_fraction": s.acceptance_fraction}), flush=True)
        s.close()
        dist.barrier()
    dist.destroy_process_group()


def c5full():
    """BASELINE configs[4] AT SCALE (launch under torchrun, one rank per GPU): DREAM on the 1000-D correlated
    Gaussian (direct log-density: the reference's log(pdf) underflows at d = 1000, SURVEY.md section 0) with
    C5_PER_GPU chains per GPU (default 1.25e6: 10^7 on 8 GPUs), in the stated sub-population mode -- every GPU
    steps its chains as one island (pairs from the local opposite half, no replica of the 80 GB population),
    islands re-dealt with one all-to-all every k generations (default 10).  History off, running moments and CR
    adaptation on.  Reports chain-steps/s (device events, max over ranks, re-deal included), the FP64-roof
    fraction of the quadratic-form kernel (2 d^2 flop per chain-step against the measured 36.5 TFLOP/s,
    profiles/r1_fp64_probe_b200.txt), acceptance and the R-hat trend from the streaming moments."""
    import ctypes as C
    import torch.distributed as dist
    from bipymc_b200 import DreamMpi, targets, _lib
    rank, local = int(os.environ["RANK"]), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    world = dist.get_world_size()
    per = int(float(os.environ.get("C5_PER_GPU", "1250000")))
    k = int(os.environ.get("C5_K", "10"))
    gens = int(os.environ.get("C5_GENS", "10"))
    N, d, warm = per * world, 1000, 3
    t = targets.Gauss_100D(dim=d)
    np.random.seed(1)
    s = DreamMpi(t.ln_like, np.zeros(d), n_chains=N, seed=3, varepsilon=np.arange(d) + 1.0, history="none",
                 burnin_gen=10 ** 6, n_cr_gen=2, device=local, subpop_k=k, device_init=True)
    done = 0
    trend = []

    def gens_run(n):
        nonlocal done
        s.run_mcmc(N * (n + 1), _k_gen0=done)
        done += n

    def note():
        rh = s.rhat()
        trend.append({"generation": done, "rhat_max": float(np.max(rh)), "rhat_median": float(np.median(rh))})

    gens_run(warm)
    note()
    _lib.check(s._libh.bpm_profile(s._handle, 1))
    torch.cuda.synchronize(); dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    gens_run(gens)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_k, n_k = (C.c_double * 8)(), (C.c_int64 * 8)()
    _lib.check(s._libh.bpm_profile_read(s._handle, ms_k, n_k))
    _lib.check(s._libh.bpm_profile(s._handle, 0))
    acc = s.acceptance_fraction
    note()
    gens_run(gens)
    note()
    mem = torch.cuda.max_memory_allocated() / 2 ** 30
    if rank == 0:
        kinds = ["split", "propose", "likelihood", "accept", "fused_phase", "cr_reduce"]
        kms = dict((kinds[i], ms_k[i] / max(1, n_k[i])) for i in range(6) if n_k[i])
        chains_per_launch = per / 2.0
        out = {"config": "C5: DREAM Gauss_1000D, %d GPUs x %d chains, sub-population mode k=%d" % (world, per, k),
               "n_chains": N, "dim": d, "generations_timed": gens,
               "chain_steps_per_s": N * gens / (float(ms.item()) * 1e-3), "ms_per_generation": float(ms.item()) / gens,
               "acceptance_fraction": acc, "rhat_trend": trend, "avg_launch_ms_by_kernel": kms,
               "redeals": getattr(s, "n_redeals", 0), "redeal_seconds_total": getattr(s, "redeal_seconds", 0.0),
               "torch_peak_alloc_GiB_per_gpu": mem}
        if "likelihood" in kms:
            tf = 2.0 * d * d * chains_per_launch / (kms["likelihood"] * 1e-3) / 1e12
            out["quadratic_form_fp64_tflops"] = tf
            out["frac_of_fp64_peak_36.5"] = tf / 36.5
            tot = sum(ms_k[i] for i in range(6))
            out["quadratic_form_share_of_kernel_time"] = ms_k[2] / tot
        print(json.dumps(out), flush=True)
    s.close()
    dist.barrier()
    dist.destroy_process_group()


def c4multi():
    """BASELINE configs[3] (launch under torchrun, 1 / 2 / 4 ranks): DREAM on the examples/ex_para_fit.py line
    fit (3 parameters, 50 data points, likelihood evaluated in-kernel), 10^5 chains in TOTAL sharded over the
    GPUs (the config as stated: strong scaling) and 10^5 chains PER GPU (weak scaling).  Per-phase fused d <= 4
    kernels; several ranks store accepted rows into the peer replicas and put the peer-memory barrier / CR exchange
    between the half-phases."""
    import torch.distributed as dist
    from bipymc_b200 import DreamMpi, targets
    rank, local = int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    world = int(os.environ.get("WORLD_SIZE", 1))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    t = targets.LineFit()
    gens, warm = 200, 20
    for label, N in (("1e5 chains in total", 100000 // world * world), ("1e5 chains per GPU", 100000 * world)):
        np.random.seed(1)
        s = DreamMpi(t.ln_like, [-0.8, 4.5, 0.2], n_chains=N, seed=3, varepsilon=1e-2, history="none",
                     burnin_gen=10 ** 6, n_cr_gen=10, device=local)
        s.run_mcmc(N * (warm + 1))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        s.run_mcmc(N * (gens + 1), _k_gen0=warm)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        if rank == 0:
            print(json.dumps({"config": "C4 linefit DREAM, %d GPU(s), %s" % (world, label), "n_gpus": world,
                              "n_chains": N, "chain_steps_per_s": N * gens / (float(ms.item()) * 1e-3),
                              "us_per_generation": 1e3 * float(ms.item()) / gens,
                              "acceptance_fraction": s.acceptance_fraction,
                              "path": "per-phase kernels" if world == 1 else
                                      "per-phase kernels + peer-memory barrier (%s)" % ("on" if s._sync_on else "off")}),
                  flush=True)
        s.close()
        if world > 1:
            dist.barrier()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    if sys.argv[1:] == ["c4multi"]:
        c4multi()
        sys.exit(0)
    if sys.argv[1:] == ["c5full"]:
        c5full()
        sys.exit(0)
    if sys.argv[1:] == ["c5multi"]:
        c5multi()
        sys.exit(0)
    if "c5shape" in (sys.argv[1:] or ["c5shape"]):
        c5shape()
        if sys.argv[1:] == ["c5shape"]:
            sys.exit(0)
    main()
