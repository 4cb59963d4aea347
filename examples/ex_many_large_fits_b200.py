#!/usr/bin/env python
"""200 relaxation-curve fits of 10^5 points each in ONE sampler: the model of examples/ex_exp_fit.py written per
observation (targets.CudaSumLikelihoodSet), each record an independent problem with its own chains, partners,
crossover adaptation and data.  Every chain's sum over its record is spread across the GPU, and all records advance
in the same kernel launches.  The fitted parameters are compared with the values the records were drawn from.

    python examples/ex_many_large_fits_b200.py
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bipymc_b200 import DreamMpi, targets  # noqa: E402

# theta = (tau, c_inf, c_0, leak, sigma): y = c_inf - c_0 exp(-t / tau) - leak t, noise of variance sigma;
# row = (t, y)
SOURCE = r'''
__device__ double ln_like_term(const double* th, const double* row) {
  const double m = th[1] + th[2] * -1.0 * exp(-row[0] / th[0]) - th[3] * row[0];
  const double r = m - row[1];
  return -0.5 * (r * r / th[4] - log(1.0 / th[4]));
}
__device__ double ln_prior(const double* th) {
  return (1.0 < th[0] && th[0] < 50.0 && -5.0 < th[1] && th[1] < 5.0 && -1.0 < th[2] && th[2] < 1.0 &&
          -5.0 < th[3] && th[3] < 5.0 && 0.0 < th[4] && th[4] < 1.0) ? 0.0 : -INFINITY;
}
'''
NAMES = ("tau", "c_inf", "c_0", "leak", "sigma")


def main(P=200, M=100000, n_chains=32, generations=1500):
    rs = np.random.RandomState(0)
    truth = np.stack([rs.uniform(5.0, 30.0, P), rs.uniform(1.0, 2.0, P), rs.uniform(0.3, 0.9, P),
                      rs.uniform(0.0, 2e-3, P), np.full(P, 2e-3)], axis=1)
    t = np.linspace(0.5, 60.0, M)
    y = (truth[:, 1:2] - truth[:, 2:3] * np.exp(-t[None] / truth[:, 0:1]) - truth[:, 3:4] * t[None] +
         np.sqrt(truth[:, 4:5]) * rs.randn(P, M))
    lik = targets.CudaSumLikelihoodSet(SOURCE, 5, np.stack([np.broadcast_to(t, (P, M)), y], axis=2), prior=True)

    # every record starts from a guess 2 % off its truth, chains in a ball of 1 % around it
    guess = truth * (1.0 + 0.02 * rs.randn(P, 5))
    np.random.seed(1)
    sampler = DreamMpi(None, guess, n_chains=n_chains, ln_like_cuda=lik, seed=7, burnin_gen=generations // 2,
                       varepsilon=(0.01 * np.abs(guess).mean(axis=0)) ** 2)
    half = generations // 2
    sampler.run_mcmc(n_chains * (half + 1))                                 # burn-in
    sampler.reset_moments()                                                 # R-hat of what follows only
    sampler.run_mcmc(n_chains * (generations - half))
    mean, std, _ = sampler.param_est(n_chains * (half + 1))                 # [P, 5] each

    z = (mean - truth) / std
    print("records: %d of %d points, chains per record: %d, generations: %d" % (P, M, n_chains, generations))
    print("acceptance fraction: median %.3f" % np.median(sampler.acceptance_fraction))
    rhat = sampler.rhat()                                                   # [P, 5]
    # a multi-problem sampler has no outlier-chain reset: a record can keep a stray chain, which R-hat shows
    print("R-hat after burn-in: median %.3f, max %.3f; records with every R-hat below 1.2: %d of %d"
          % (np.median(rhat), rhat.max(), np.sum(np.all(rhat < 1.2, axis=1)), P))
    for q, name in enumerate(NAMES):
        print("%-6s |fit - truth| / posterior sd: median %.2f, 95th percentile %.2f; truths inside the 95%% "
              "credible interval: %.3f" % (name, np.median(np.abs(z[:, q])), np.percentile(np.abs(z[:, q]), 95),
                                           np.mean(np.abs(z[:, q]) < 1.96)))
    for g in range(2):
        print("record %d: " % g + ", ".join("%s = %.5g +- %.2g (true %.5g)" % (NAMES[q], mean[g, q], std[g, q],
                                                                              truth[g, q]) for q in range(5)))


if __name__ == "__main__":
    main()
