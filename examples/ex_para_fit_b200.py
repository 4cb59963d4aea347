#!/usr/bin/env python
"""Line fit with a nuisance scatter parameter -- the workload of the reference's
examples/ex_para_fit.py (theta = (m, b, ln f), 50 synthetic points, box prior), run four ways
on the device sampler:

  1. the built-in device likelihood (whole generations inside the CUDA kernels),
  2. the reference's per-term likelihood as CUDA source (targets.CudaLikelihood, compiled at run
     time into the same kernels; fmad=False rounds every operation like numpy),
  3. a batched torch likelihood  f(theta[n, 3]) -> lnL[n]  (device tensors, same stream),
  4. the reference's scalar ln_like_fn(theta, x, y, yerr) with ln_kwargs (host round trip).

Usage:  python examples/ex_para_fit_b200.py            (one GPU)
        torchrun --nproc-per-node 2 examples/ex_para_fit_b200.py   (chains sharded over 2 GPUs)
"""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# ex_para_fit.py:39-55, one data point at a time; data = x[M], y[M], yerr[M]
LNPROB_CUDA = r'''
__device__ double ln_like(const double* theta, const double* data) {
  const int M = BPM_NDATA / 3;
  const double* x = data;
  const double* y = data + M;
  const double* yerr = data + 2 * M;
  const double m = theta[0], b = theta[1], lnf = theta[2];
  if (!(-5.0 < m && m < 0.5 && 0.0 < b && b < 10.0 && -10.0 < lnf && lnf < 1.0)) return -INFINITY;
  const double e2 = exp(2.0 * lnf);
  double s = 0.0;
  for (int i = 0; i < M; ++i) {
    const double model = m * x[i] + b;
    const double inv_sigma2 = 1.0 / (yerr[i] * yerr[i] + model * model * e2);
    s += (y[i] - model) * (y[i] - model) * inv_sigma2 - log(inv_sigma2);
  }
  return 0.0 + -0.5 * s;
}
'''


def make_lnprob_batched(x, y, yerr):
    """The same likelihood as torch ops on [n, 3] CUDA float64 tensors (x, y, yerr: CUDA tensors)."""
    import torch

    def lnprob_batched(theta):
        m, b, lnf = theta[:, 0:1], theta[:, 1:2], theta[:, 2:3]
        model = m * x[None, :] + b
        inv_sigma2 = 1.0 / (yerr[None, :] ** 2 + model ** 2 * torch.exp(2 * lnf))
        ll = -0.5 * ((y[None, :] - model) ** 2 * inv_sigma2 - torch.log(inv_sigma2)).sum(dim=1)
        ok = (theta[:, 0] > -5.0) & (theta[:, 0] < 0.5) & (theta[:, 1] > 0.0) & (theta[:, 1] < 10.0) & \
             (theta[:, 2] > -10.0) & (theta[:, 2] < 1.0)
        return torch.where(ok, ll, torch.full_like(ll, -float("inf")))
    return lnprob_batched


def main():
    import torch
    from bipymc_b200 import DreamMpi, targets
    if "RANK" in os.environ:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist.init_process_group("nccl")
    rank = int(os.environ.get("RANK", 0))
    fit = targets.LineFit()                         # x, y, yerr generated like ex_para_fit.py:17,26-35
    theta_0 = np.array([-0.8, 4.5, 0.2])
    lnprob_batched = make_lnprob_batched(*(torch.from_numpy(v).cuda() for v in (fit.x, fit.y, fit.yerr)))
    lik = targets.CudaLikelihood(LNPROB_CUDA, 3, np.concatenate([fit.x, fit.y, fit.yerr]), fmad=False)

    def lnprob_scalar(theta, x, y, yerr):           # the reference's plug-in signature (samplers.py:36-43)
        return targets.LineFit(x, y, yerr).ln_like(theta)

    runs = [("device target", dict(ln=fit.ln_like), 20000, 300),
            ("CUDA source plug-in", dict(ln=lnprob_scalar, ln_like_cuda=lik,
                                         ln_kwargs=dict(x=fit.x, y=fit.y, yerr=fit.yerr)), 20000, 300),
            ("batched torch plug-in", dict(ln=lnprob_scalar, ln_like_batched=lnprob_batched,
                                           ln_kwargs=dict(x=fit.x, y=fit.y, yerr=fit.yerr)), 20000, 300),
            ("scalar host plug-in", dict(ln=lnprob_scalar, ln_kwargs=dict(x=fit.x, y=fit.y, yerr=fit.yerr)), 64, 300)]
    for name, kw, n_chains, gens in runs:
        np.random.seed(42)
        ln = kw.pop("ln")
        s = DreamMpi(ln, theta_0, n_chains=n_chains, varepsilon=1e-4, n_cr_gen=50, burnin_gen=150, seed=1,
                     history="full", **kw)
        t0 = time.perf_counter()
        s.run_mcmc(n_chains * (gens + 1))
        dt = time.perf_counter() - t0
        mean, std, _ = s.param_est(n_burn=n_chains * (gens // 2))
        if rank == 0:
            print("%-22s %6d chains x %d generations  %.2f s   m = %.3f +- %.3f  b = %.3f +- %.3f  ln f = %.3f +- %.3f"
                  "   acc %.2f  R-hat %s" % (name, n_chains, gens, dt, mean[0], std[0], mean[1], std[1], mean[2], std[2],
                                             s.acceptance_fraction, np.round(s.rhat(), 3)))
        s.close()


if __name__ == "__main__":
    main()
