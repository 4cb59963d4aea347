#!/usr/bin/env python
"""The exp model of the reference's examples/ex_exp_fit.py fitted to 10^5 observations with 1024 DREAM
chains, the likelihood written once per observation (targets.CudaSumLikelihood: every chain's sum is
spread over the whole GPU) and once as a whole function (targets.CudaLikelihood: one thread per chain
walks all observations).  Both give the same posterior; the sum form is the one that fills the GPU
when there are few chains and many observations.

    python examples/ex_large_data_fit_b200.py [n_obs] [n_gen]"""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from bipymc_b200 import DreamMpi, targets  # noqa: E402

# ex_exp_fit.py:38-43, 73-121: theta = (tau, c_inf, c_0, leak, sigma), box prior
PRIOR = r'''
__device__ double ln_prior(const double* th) {
  const double tau = th[0], c_inf = th[1], c_0 = th[2], leak = th[3], sigma = th[4];
  return (-5.0 < c_inf && c_inf < 5.0 && 1.0 < tau && tau < 50.0 && -1.0 < c_0 && c_0 < 1.0 &&
          -5.0 < leak && leak < 5.0 && 0.0 < sigma && sigma < 1.0) ? 0.0 : -INFINITY;
}
'''
TERM = r'''
__device__ double ln_like_term(const double* th, const double* row) {   // row = (t, y)
  const double m = th[1] + th[2] * -1.0 * exp(-row[0] / th[0]) - th[3] * row[0];
  return -0.5 * ((m - row[1]) * (m - row[1]) / th[4] - log(1.0 / th[4]));
}
'''
WHOLE = r'''
__device__ double ln_like(const double* th, const double* data) {        // data = t[M], y[M]
  const int M = BPM_NDATA / 2;
  const double tau = th[0], c_inf = th[1], c_0 = th[2], leak = th[3], sigma = th[4];
  if (!(-5.0 < c_inf && c_inf < 5.0 && 1.0 < tau && tau < 50.0 && -1.0 < c_0 && c_0 < 1.0 &&
        -5.0 < leak && leak < 5.0 && 0.0 < sigma && sigma < 1.0)) return -INFINITY;
  double s = 0.0;
  for (int i = 0; i < M; ++i) {
    const double m = c_inf + c_0 * -1.0 * exp(-data[i] / tau) - leak * data[i];
    s += -0.5 * ((m - data[M + i]) * (m - data[M + i]) / sigma - log(1.0 / sigma));
  }
  return s;
}
'''


def fit(lik, n_chains, n_gen):
    import torch
    np.random.seed(42)
    s = DreamMpi(targets.ExpFit().ln_like, [12.0, 1.5, 0.6, 1e-3, 2e-3], n_chains=n_chains, seed=7,
                 varepsilon=np.asarray([1e-2, 1e-2, 1e-3, 1e-8, 1e-9]) * 1e-2, ln_like_cuda=lik,
                 burnin_gen=n_gen // 2, n_cr_gen=10)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s.run_mcmc(n_chains * (n_gen + 1))
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    post = s._hist.tensor()[n_gen // 2:, :, :5].cpu().numpy().reshape(-1, 5)
    return post, dt / n_gen


def main():
    n_obs = int(sys.argv[1]) if len(sys.argv) > 1 else 100000
    n_gen = int(sys.argv[2]) if len(sys.argv) > 2 else 200
    t, y = targets.expfit_data(n=n_obs)
    forms = [("per observation (CudaSumLikelihood)",
              targets.CudaSumLikelihood(TERM + PRIOR, 5, np.stack([t, y], axis=1), prior=True)),
             ("whole function (CudaLikelihood)", targets.CudaLikelihood(WHOLE, 5, np.concatenate([t, y])))]
    names = ["tau", "c_inf", "c_0", "leak", "sigma"]
    for label, lik in forms:
        post, per_gen = fit(lik, 1024, n_gen)
        print("%s: %.3f ms per generation" % (label, per_gen * 1e3))
        for i, nm in enumerate(names):
            print("  %-6s %.6g +- %.3g" % (nm, post[:, i].mean(), post[:, i].std()))


if __name__ == "__main__":
    main()
