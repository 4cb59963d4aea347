"""Gaussian likelihood with a dense data covariance: ms per DREAM generation, the likelihood's share of it and its
useful FP64 rate, for three ways of running the same likelihood.

Workload: DREAM on the exp model (d = 4: tau, c_inf, c_0, leak) with exponential-kernel noise over M times, for N
chains.  Arms, run alternately, each repeated:
  gauss  -- targets.CudaGaussLikelihood (model kernel, DMMA quadratic form with triangular skip, finish);
  whole  -- targets.CudaLikelihood whose ln_like loops over B = L^-T in data, one thread per chain (only at the
            sizes where it finishes in reasonable time);
  torch  -- ln_like_batched with torch.matmul against B.
The useful work of one half-phase is n M (M + 1) flop, n = N / 2: the upper triangle of (m - y) B and its squares.
Writes one JSON line per (arm, N, M, repeat), plus the card's name and power limit, to --out.

    python tools/gauss_likelihood_bench.py --out DIR [--gens 30] [--repeats 2]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

MEAN = r'''
__device__ double model_mean(const double* th, const double* row) {
  return th[1] + th[2] * -1.0 * exp(-row[0] / th[0]) - th[3] * row[0];
}
'''
PRIOR = r'''
__device__ double ln_prior(const double* th) {
  return (1.0 < th[0] && th[0] < 50.0 && -5.0 < th[1] && th[1] < 5.0 && -1.0 < th[2] && th[2] < 1.0 &&
          -5.0 < th[3] && th[3] < 5.0) ? 0.0 : -INFINITY;
}
'''
# the whole-function form: data = (t[M], y[M], B[M][M])
WHOLE = r'''
__device__ double ln_like(const double* th, const double* data) {
  if (!(1.0 < th[0] && th[0] < 50.0 && -5.0 < th[1] && th[1] < 5.0 && -1.0 < th[2] && th[2] < 1.0 &&
        -5.0 < th[3] && th[3] < 5.0)) return -INFINITY;
  const int M = BPM_NDATA_M;
  const double* t = data;
  const double* y = data + M;
  const double* B = data + 2 * M;
  double r[BPM_NDATA_M];
  for (int k = 0; k < M; ++k) r[k] = th[1] + th[2] * -1.0 * exp(-t[k] / th[0]) - th[3] * t[k] - y[k];
  double maha = 0.0;
  for (int j = 0; j < M; ++j) {
    double z = 0.0;
    for (int k = 0; k <= j; ++k) z += r[k] * B[(size_t)k * M + j];
    maha += z * z;
  }
  return -0.5 * (BPM_C0 + maha);
}
'''
THETA = np.array([12.0, 1.5, 0.6, 1e-3])


def problem(M, seed=0):
    t = np.linspace(0.5, 60.0, M)
    cov = 0.02 ** 2 * np.exp(-np.abs(t[:, None] - t[None, :]) / 5.0) + 1e-6 * np.eye(M)
    m = THETA[1] + THETA[2] * -1.0 * np.exp(-t / THETA[0]) - THETA[3] * t
    y = m + np.linalg.cholesky(cov) @ np.random.RandomState(seed).randn(M)
    return t, y, cov


def make(arm, N, t, y, cov, gauss_lik):
    import torch
    from bipymc_b200 import DreamMpi, targets
    kw = dict(n_chains=N, seed=5, varepsilon=np.array([1e-2, 1e-4, 1e-4, 1e-8]), n_cr_gen=3, burnin_gen=10 ** 6,
              history="none")
    M = t.size
    never = lambda th: 0.0                                                  # noqa: E731
    if arm == "gauss":
        return DreamMpi(never, THETA, ln_like_cuda=gauss_lik, **kw)
    B, c0 = gauss_lik.B, gauss_lik.c0
    if arm == "whole":
        src = "#define BPM_NDATA_M %d\n#define BPM_C0 %.17g\n" % (M, c0) + WHOLE
        lik = targets.CudaLikelihood(src, 4, np.concatenate([t, y, B.ravel()]))
        return DreamMpi(never, THETA, ln_like_cuda=lik, **kw)
    dev = torch.device("cuda", torch.cuda.current_device())
    tt, yt, Bt = (torch.from_numpy(a).to(dev) for a in (t, y, B))

    def batched(th):
        m = th[:, 1:2] + th[:, 2:3] * -1.0 * torch.exp(-tt[None, :] / th[:, 0:1]) - th[:, 3:4] * tt[None, :]
        z = torch.matmul(m - yt[None, :], Bt)
        v = -0.5 * (c0 + (z * z).sum(dim=1))
        ok = (th[:, 0] > 1) & (th[:, 0] < 50) & (th[:, 1].abs() < 5) & (th[:, 2].abs() < 1) & (th[:, 3].abs() < 5)
        return torch.where(ok, v, torch.full_like(v, -float("inf")))
    return DreamMpi(never, THETA, ln_like_batched=batched, **kw)


def timed(s, N, gens):
    """ms per generation over `gens` generations (device synchronised), then the likelihood record's share and ms
    from a separate profiled window of the same length."""
    import torch
    from bipymc_b200 import _lib
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s.run_mcmc(N * gens)
    torch.cuda.synchronize()
    ms_gen = 1e3 * (time.perf_counter() - t0) / gens
    share = lik_ms = None
    if s._mode() == "device":
        import ctypes as C
        _lib.check(s._libh.bpm_profile(s._handle, 1))
        s.run_mcmc(N * gens)
        ms, n = (C.c_double * 8)(), (C.c_int64 * 8)()
        _lib.check(s._libh.bpm_profile_read(s._handle, ms, n))
        _lib.check(s._libh.bpm_profile(s._handle, 0))
        lik_ms = ms[2] / gens
        share = ms[2] / sum(ms)
    return ms_gen, share, lik_ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--gens", type=int, default=30)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--N", type=int, nargs="*", default=[1024, 10000])
    ap.add_argument("--M", type=int, nargs="*", default=[256, 1024, 4096])
    ap.add_argument("--whole-max-m", type=int, default=1024, help="largest M the whole-function arm runs at")
    a = ap.parse_args()
    import torch
    from bipymc_b200 import targets
    assert torch.cuda.is_available(), "this benchmark measures the GPU and needs one"
    os.makedirs(a.out, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    with open(os.path.join(a.out, "gpu.txt"), "w") as f:
        f.write(gpu + "\n")
    out = open(os.path.join(a.out, "gauss_likelihood_bench.jsonl"), "w")
    for M in a.M:
        t, y, cov = problem(M)
        lik = targets.CudaGaussLikelihood(MEAN + PRIOR, 4, t, y, cov, prior=True)
        for N in a.N:
            arms = ["gauss", "torch"] + (["whole"] if M <= a.whole_max_m else [])
            samplers = {arm: make(arm, N, t, y, cov, lik) for arm in arms}
            for arm in arms:                                               # warm-up: modules, algorithms
                samplers[arm].run_mcmc(N * 5)
            for rep in range(a.repeats):
                for arm in arms:                                           # alternate the arms
                    gens = a.gens if arm != "whole" else max(3, a.gens // 10)
                    ms_gen, share, lik_ms = timed(samplers[arm], N, gens)
                    flop = 2 * (N // 2) * M * (M + 1)                        # two half-phases of n M (M + 1)
                    rec = dict(arm=arm, N=N, M=M, rep=rep, gens=gens, ms_per_gen=ms_gen, lik_share=share,
                               lik_ms_per_gen=lik_ms,
                               lik_tflops=(flop / (lik_ms * 1e-3) / 1e12) if lik_ms else None,
                               e2e_tflops=flop / (ms_gen * 1e-3) / 1e12, gpu=gpu)
                    if lik_ms:
                        rec["share_of_dmma_peak_36_9"] = rec["lik_tflops"] / 36.9
                    print(json.dumps(rec), flush=True)
                    out.write(json.dumps(rec) + "\n")
                    out.flush()
            del samplers
            torch.cuda.empty_cache()
    out.close()


if __name__ == "__main__":
    main()
