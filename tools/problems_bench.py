#!/usr/bin/env python
"""Many fits in one sampler (targets.CudaLikelihoodSet): time per generation of multi-problem DREAM runs, the
fused / split kernels' share from bpm_profile_read, and what users do without it -- one CudaLikelihood sampler per
problem, one after another.  CUDA events around whole run_mcmc calls after a warm-up run of the same shape;
the profile is taken in a run of its own.  Prints one JSON line per case, the first one naming the card and its
power limit.

    python tools/problems_bench.py [--gens 200] [--warmup 20] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from test_cuda_likelihood_cpu import LINEFIT_PER_TERM  # noqa: E402

# the reference's exp fit (examples/ex_exp_fit.py:73-121) in its per-term form; data = t[M], y[M]
EXPFIT_PER_TERM = r'''
__device__ double ln_like(const double* th, const double* data) {
  const int M = BPM_NDATA / 2;
  const double tau = th[0], c_inf = th[1], c_0 = th[2], leak = th[3], sigma = th[4];
  if (!(-5.0 < c_inf && c_inf < 5.0 && 1.0 < tau && tau < 50.0 && -1.0 < c_0 && c_0 < 1.0 && -5.0 < leak &&
        leak < 5.0 && 0.0 < sigma && sigma < 1.0)) return -INFINITY;
  double s = 0.0;
  for (int i = 0; i < M; ++i) {
    const double m = c_inf + c_0 * -1.0 * exp(-data[i] / tau) - leak * data[i];
    const double r = m - data[M + i];
    s += r * r / sigma - log(1.0 / sigma);
  }
  return 0.0 + -0.5 * s;
}
'''
KINDS = ("split", "propose", "likelihood", "accept", "fused_phase", "cr_reduce")


def _never(theta, **kw):
    raise AssertionError("not called")


def linefit_rows(P, seed=0):
    from bipymc_b200 import targets
    x, y, yerr = targets.linefit_data(n=50)
    rs = np.random.RandomState(seed)
    rows = np.tile(np.concatenate([x, y, yerr]), (P, 1))
    rows[:, 50:100] = rows[:, 50:100] * (1.0 + 0.05 * rs.randn(P, 1)) + 0.2 * rs.randn(P, 1)
    return rows


def expfit_rows(P, seed=0):
    from bipymc_b200 import targets
    t, y = targets.expfit_data(n=60)
    rs = np.random.RandomState(seed)
    rows = np.tile(np.concatenate([t, y]), (P, 1))
    rows[:, 60:] += 0.01 * rs.randn(P, 1)
    return rows


def sampler(lik, theta0, n, var):
    from bipymc_b200 import DreamMpi
    np.random.seed(1)
    return DreamMpi(_never, np.asarray(theta0, dtype=float), n_chains=n, seed=3, ln_like_cuda=lik, varepsilon=var,
                    n_cr_gen=10, burnin_gen=100000)


def run_timed(samplers, n, gens):
    """Milliseconds of `gens` generations of every sampler in turn (CUDA events, one stream)."""
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for s in samplers:
        s.run_mcmc(n * (gens + 1))
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def profile(s, n, gens):
    from bipymc_b200 import _lib
    _lib.check(s._libh.bpm_profile(s._handle, 1))
    s.run_mcmc(n * (gens + 1))
    ms, cnt = (C.c_double * 8)(), (C.c_int64 * 8)()
    _lib.check(s._libh.bpm_profile_read(s._handle, ms, cnt))
    _lib.check(s._libh.bpm_profile(s._handle, 0))
    return {k: dict(launches_per_gen=cnt[i] / gens, us_per_launch=round(1e3 * ms[i] / cnt[i], 2) if cnt[i] else 0.0)
            for i, k in enumerate(KINDS) if cnt[i]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gens", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from bipymc_b200 import targets
    if not torch.cuda.is_available():
        raise SystemExit("problems_bench.py needs a CUDA device")
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
    emit(dict(gpu=torch.cuda.get_device_name(0), nvidia_smi=q, gens=args.gens, warmup=args.warmup))
    G, W = args.gens, args.warmup
    cases = [("linefit P=1000 n=100 M=50", LINEFIT_PER_TERM, 3, linefit_rows, 1000, 100, [-0.9, 4.3, -0.7], 1e-3),
             ("linefit P=10000 n=32 M=50", LINEFIT_PER_TERM, 3, linefit_rows, 10000, 32, [-0.9, 4.3, -0.7], 1e-3),
             ("expfit d=5 P=1000 n=100 M=60", EXPFIT_PER_TERM, 5, expfit_rows, 1000, 100,
              [12.0, 1.5, 0.6, 1e-3, 2e-3], 1e-8)]
    for name, src, d, rows_fn, P, n, th, var in cases:
        lik = targets.CudaLikelihoodSet(src, d, rows_fn(P), fmad=False)
        s = sampler(lik, th, n, var)
        run_timed([s], n, W)
        ms = run_timed([s], n, G)
        emit(dict(case=name, chains=P * n, us_per_generation=round(1e3 * ms / G, 2),
                  us_per_problem_generation=round(1e3 * ms / G / P, 4), profile=profile(s, n, G)))
        del s
    # the same model as ONE population of 10^5 chains (single-problem CudaLikelihood), for comparison
    lik = targets.CudaLikelihood(LINEFIT_PER_TERM, 3, linefit_rows(1)[0], fmad=False)
    s = sampler(lik, [-0.9, 4.3, -0.7], 100000, 1e-3)
    run_timed([s], 100000, W)
    ms = run_timed([s], 100000, G)
    emit(dict(case="linefit one population of 10^5 chains", chains=100000, us_per_generation=round(1e3 * ms / G, 2),
              profile=profile(s, 100000, G)))
    del s
    # what users do today: one CudaLikelihood sampler per problem, run one after another
    rows = linefit_rows(32)
    ss = [sampler(targets.CudaLikelihood(LINEFIT_PER_TERM, 3, rows[g], fmad=False), [-0.9, 4.3, -0.7], 100, 1e-3)
          for g in range(32)]
    run_timed(ss, 100, W)
    ms = run_timed(ss, 100, G)
    emit(dict(case="linefit separate samplers, 32 problems x n=100, one after another", chains=3200,
              us_per_problem_generation=round(1e3 * ms / G / 32, 2)))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
