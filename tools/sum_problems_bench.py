#!/usr/bin/env python
"""Many datasets of many observations in one sampler (targets.CudaSumLikelihoodSet): time per generation of
multi-problem DREAM runs, the likelihood launch's share and terms/s from bpm_profile_read, against the same data as
a CudaLikelihoodSet (whole function, one thread per chain) and as separate CudaSumLikelihood samplers run one after
another.  The model is the reference's exp fit (examples/ex_exp_fit.py:73-121) per observation, fmad=False.
Timing and profile as in problems_bench.py: CUDA events around whole run_mcmc calls after a warm-up run of the
same shape; the profile in a run of its own.  Prints one JSON line per measurement, the first naming the card and
its power limit.

    python tools/sum_problems_bench.py [--out FILE]
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

from problems_bench import EXPFIT_PER_TERM, profile, run_timed, sampler  # noqa: E402
from test_cuda_sum_likelihood_cpu import EXPFIT_PRIOR, EXPFIT_TERM  # noqa: E402

THETA0 = [12.0, 1.5, 0.6, 1e-3, 2e-3]
VAR = 1e-8
# (P, n, M, generations of the set forms, of the whole-function set, separate samplers run, their generations)
CASES = [(100, 32, 100000, 50, 3, 100, 5), (1000, 64, 1000, 200, 20, 100, 20)]


def expfit_set(P, M, seed=0):
    """[P][M][2] rows (t, y): the synthetic exp-fit series with the ordinate shifted per problem."""
    from bipymc_b200 import targets
    t, y = targets.expfit_data(n=M)
    rs = np.random.RandomState(seed)
    rows = np.empty((P, M, 2))
    rows[:, :, 0] = t
    rows[:, :, 1] = y[None] + 0.01 * rs.randn(P, 1)
    return rows


def measure(s, n, P, M, gens, warmup):
    """us per generation (timed run) and the likelihood launch's share and terms/s (profiled run)."""
    run_timed([s], n, warmup)
    ms = run_timed([s], n, gens)
    prof = profile(s, n, gens)
    tot = sum(v["launches_per_gen"] * v["us_per_launch"] for v in prof.values())
    lk = prof["likelihood"]["launches_per_gen"] * prof["likelihood"]["us_per_launch"]
    return dict(us_per_generation=round(1e3 * ms / gens, 2), us_per_problem_generation=round(1e3 * ms / gens / P, 4),
                likelihood_share=round(lk / tot, 4), likelihood_us_per_gen=round(lk, 2),
                terms_per_s=float("%.4g" % (P * n * M / (lk * 1e-6))), profile=prof)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from bipymc_b200 import targets
    if not torch.cuda.is_available():
        raise SystemExit("sum_problems_bench.py needs a CUDA device")
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
    for P, n, M, gens, gens_whole, n_sep, gens_sep in CASES:
        rows = expfit_set(P, M)
        shape = dict(P=P, n=n, M=M, k=2)
        s = sampler(targets.CudaSumLikelihoodSet(EXPFIT_TERM + EXPFIT_PRIOR, 5, rows, prior=True, fmad=False),
                    THETA0, n, VAR)
        emit(dict(case="CudaSumLikelihoodSet", gens=gens, **shape, **measure(s, n, P, M, gens, gens // 10)))
        del s
        whole = np.concatenate([rows[:, :, 0], rows[:, :, 1]], axis=1)          # t[M], y[M] per problem
        s = sampler(targets.CudaLikelihoodSet(EXPFIT_PER_TERM, 5, whole, fmad=False), THETA0, n, VAR)
        emit(dict(case="CudaLikelihoodSet (whole function)", gens=gens_whole, **shape,
                  **measure(s, n, P, M, gens_whole, 2)))
        del s
        # what users do without the set: one CudaSumLikelihood sampler per problem, run one after another
        ss = [sampler(targets.CudaSumLikelihood(EXPFIT_TERM + EXPFIT_PRIOR, 5, rows[q], prior=True, fmad=False),
                      THETA0, n, VAR) for q in range(n_sep)]
        run_timed(ss, n, 2)
        ms = run_timed(ss, n, gens_sep)
        emit(dict(case="separate CudaSumLikelihood samplers, one after another", problems_run=n_sep,
                  gens=gens_sep, **shape, us_per_problem_generation=round(1e3 * ms / gens_sep / n_sep, 2)))
        del ss
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
