#!/usr/bin/env python
"""Many datasets of different lengths in one sampler (targets.CudaSumLikelihoodSet given a list of arrays): time per
generation of multi-problem DREAM runs, the likelihood launch's share and useful terms/s (sum_g M_g times the chains
evaluated, over the likelihood launches' time), against the same data padded to the longest dataset with a mask
column as a rectangular CudaSumLikelihoodSet, and against separate CudaSumLikelihood samplers run one after another.
The model is the reference's exp fit (examples/ex_exp_fit.py:73-121) per observation with its box prior,
fmad=False.  Timing and profile as in sum_problems_bench.py: CUDA events around whole run_mcmc calls after a
warm-up run of the same shape; the profile in a run of its own.  Prints one JSON line per measurement, the first
naming the card and its power limit.

    python tools/sum_ragged_bench.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))

from problems_bench import run_timed, sampler  # noqa: E402
from sum_problems_bench import THETA0, VAR, measure  # noqa: E402
from test_cuda_sum_likelihood_cpu import EXPFIT_PRIOR, EXPFIT_TERM  # noqa: E402

# the padded form's term: rows (t, y, mask), mask 0.0 on the padding
EXPFIT_MASKED_TERM = r'''
__device__ double ln_like_term(const double* th, const double* row) {
  if (row[2] == 0.0) return 0.0;
  const double m = th[1] + th[2] * -1.0 * exp(-row[0] / th[0]) - th[3] * row[0];
  const double r = m - row[1];
  return -0.5 * (r * r / th[4] - log(1.0 / th[4]));
}
'''
# (name, P, n, lengths(seeded), generations of the ragged set, of the padded set, separate samplers, their generations)
CASES = [("a: M log-uniform in [1e2, 1e5]", 1000, 32,
          lambda rs, P: np.exp(rs.uniform(np.log(1e2), np.log(1e5), P)).astype(np.int64), 100, 20, 20, 10),
         ("b: M uniform in [5e4, 1e5]", 100, 32, lambda rs, P: rs.randint(50000, 100001, P).astype(np.int64),
          50, 20, 20, 10)]


def expfit_ragged(lengths, seed=0):
    """Problem g: the synthetic exp-fit series of lengths[g] rows (t, y), the ordinate shifted per problem."""
    from bipymc_b200 import targets
    rs = np.random.RandomState(seed)
    out = []
    for m in lengths:
        t, y = targets.expfit_data(n=int(m))
        out.append(np.stack([t, y + 0.01 * rs.randn()], axis=1))
    return out


def per_problem(m, P):
    """measure() of all P problems as one (its terms_per_s counts sum_g M_g rows): per problem-generation."""
    m["us_per_problem_generation"] = round(m["us_per_generation"] / P, 4)
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from bipymc_b200 import targets
    if not torch.cuda.is_available():
        raise SystemExit("sum_ragged_bench.py needs a CUDA device")
    lines = []

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        lines.append(line)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:          # the measurement stands without it, but say why it is missing
        q = "nvidia-smi unavailable: %s" % e
    emit(dict(gpu=torch.cuda.get_device_name(0), nvidia_smi=q))
    src = EXPFIT_TERM + EXPFIT_PRIOR
    for name, P, n, lengths_fn, gens, gens_pad, n_sep, gens_sep in CASES:
        lengths = lengths_fn(np.random.RandomState(7), P)
        parts = expfit_ragged(lengths)
        M_sum, M_max = int(lengths.sum()), int(lengths.max())
        shape = dict(workload=name, P=P, n=n, rows=M_sum, longest=M_max, padded_rows=P * M_max,
                     useful_over_padded=round(M_sum / (P * M_max), 4))
        s = sampler(targets.CudaSumLikelihoodSet(src, 5, parts, prior=True, fmad=False), THETA0, n, VAR)
        emit(dict(case="ragged CudaSumLikelihoodSet", gens=gens, **shape, **per_problem(
            measure(s, n, 1, M_sum, gens, gens // 10), P)))
        del s
        padded = np.zeros((P, M_max, 3))
        for g, p in enumerate(parts):
            padded[g, :p.shape[0], :2] = p
            padded[g, :p.shape[0], 2] = 1.0
        s = sampler(targets.CudaSumLikelihoodSet(EXPFIT_MASKED_TERM + EXPFIT_PRIOR, 5, padded, prior=True, fmad=False),
                    THETA0, n, VAR)
        del padded
        # terms_per_s counts the useful terms only
        emit(dict(case="rectangular CudaSumLikelihoodSet padded with a mask column", gens=gens_pad, **shape,
                  **per_problem(measure(s, n, 1, M_sum, gens_pad, 2), P)))
        del s
        ss = [sampler(targets.CudaSumLikelihood(src, 5, parts[g], prior=True, fmad=False), THETA0, n, VAR)
              for g in range(n_sep)]
        run_timed(ss, n, 2)
        ms = run_timed(ss, n, gens_sep)
        emit(dict(case="separate CudaSumLikelihood samplers, one after another", problems_run=n_sep,
                  rows_run=int(lengths[:n_sep].sum()), gens=gens_sep, **shape,
                  us_per_problem_generation=round(1e3 * ms / gens_sep / n_sep, 2)))
        del ss
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
