#!/usr/bin/env python
"""1000 straight-line fits in ONE sampler: each dataset is an independent problem with its own chains,
partners, crossover adaptation and data (targets.CudaLikelihoodSet), and all of them advance in the same
kernel launches.  The fitted slopes and intercepts are compared with the values the data were drawn from.

    python examples/ex_many_fits_b200.py
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bipymc_b200 import DreamMpi, targets  # noqa: E402

# y = a + b x, Gaussian noise of known sigma; data row = x[M], y[M], sigma[M]
SOURCE = r'''
__device__ double ln_like(const double* theta, const double* data) {
  const int M = BPM_NDATA / 3;
  if (!(fabs(theta[0]) < 100.0 && fabs(theta[1]) < 100.0)) return -INFINITY;
  double s = 0.0;
  for (int i = 0; i < M; ++i) {
    const double r = (data[M + i] - theta[0] - theta[1] * data[i]) / data[2 * M + i];
    s += r * r;
  }
  return -0.5 * s;
}
'''


def main(P=1000, M=30, n_chains=64, generations=600):
    rs = np.random.RandomState(0)
    a_true, b_true = rs.uniform(-5.0, 5.0, P), rs.uniform(-2.0, 2.0, P)
    x = np.sort(rs.uniform(0.0, 10.0, (P, M)), axis=1)
    sigma = 0.2 + 0.3 * rs.rand(P, M)
    y = a_true[:, None] + b_true[:, None] * x + sigma * rs.randn(P, M)
    lik = targets.CudaLikelihoodSet(SOURCE, 2, np.concatenate([x, y, sigma], axis=1))

    np.random.seed(1)
    sampler = DreamMpi(None, np.zeros(2), n_chains=n_chains, ln_like_cuda=lik, varepsilon=1.0, seed=7,
                       burnin_gen=generations // 2)
    sampler.run_mcmc(n_chains * (generations + 1))
    mean, std, _ = sampler.param_est(n_chains * (generations // 2))       # [P, 2] each

    z = (mean - np.stack([a_true, b_true], axis=1)) / std
    print("problems: %d, chains per problem: %d, generations: %d" % (P, n_chains, generations))
    print("acceptance fraction: median %.3f" % np.median(sampler.acceptance_fraction))
    print("max R-hat: %.3f" % sampler.rhat().max())
    print("|fit - truth| / posterior sd: median %.2f, 95th percentile %.2f" % (np.median(np.abs(z)),
                                                                              np.percentile(np.abs(z), 95)))
    print("share of truths inside the 95%% credible interval: %.3f" % np.mean(np.abs(z) < 1.96))
    for g in range(3):
        print("problem %d: a = %.3f +- %.3f (true %.3f), b = %.3f +- %.3f (true %.3f)"
              % (g, mean[g, 0], std[g, 0], a_true[g], mean[g, 1], std[g, 1], b_true[g]))


if __name__ == "__main__":
    main()
