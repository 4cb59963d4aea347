"""Run-time compiled likelihoods on the GPU at the shapes the rest of the suite never runs.

  A. sum kernels against the order contract, bit for bit (fmad=False): row lengths on both sides of every
     staging boundary and past it, d on both sides of the register / pointer theta boundary, and row counts
     that reach every launch-shape branch (test_jit_shapes_cpu.py: sum_plan), at batch sizes 1, 7 and
     >= 4096; chains outside the prior inside a CTA tile;
  B. sum kernels (fmad=True) against the correctly rounded sum, within the error bound of their tree;
  C. CudaLikelihood and CudaSumLikelihood in the generic propose / likelihood / accept kernels at
     LPC 4, 8 and 32 (d on both sides of each boundary) against the oracle step (1e-12);
  D. "problem g equals its single-problem sampler" at n = 4 .. 4099 chains per problem, d = 2 (fused),
     20 (LPC 8) and 40 (LPC 32), n_cr = 3 and 6, DREAM and DE-MC; and bpm_eval_lnl of a multi-problem
     handle against numpy, bit for bit."""
import numpy as np
import pytest

from test_cuda_sum_likelihood_cpu import CHUNK, sum_order
from test_cuda_sum_likelihood_gpu import _eval, _sampler
from test_jit_shapes_cpu import (ALLCOL_PRIOR, ALLCOL_TERM, D_CHAINS, D_DIMS, GAUSS_DIAG, LIN_TERM, ORACLE_DIMS,
                                 ORACLE_SUM, SUM_CASES, allcol_data, allcol_terms_np, gauss_diag_data, lin_exact_sum,
                                 n_problems)
from test_native_gpu import _native_vs_oracle
from test_problems_gpu import _assert_problem_equal, _multi, _single_like
from test_replay_parity_gpu import launches_by_kind

pytestmark = pytest.mark.gpu

U = 2.0 ** -53          # unit roundoff of float64


def _never(theta, **kw):
    raise AssertionError("ln_like_fn must not be called when ln_like_cuda is given")


def _thetas(n, d, seed=3):
    return np.random.RandomState(seed).uniform(-0.5, 0.5, (n, d))


# ---- A. the order contract at every launch shape ---------------------------------------------------------
@pytest.mark.parametrize("case", range(len(SUM_CASES)),
                         ids=["k%d_d%d_M%d%s" % (c[0], c[1], c[2], "_prior" if c[4] else "") for c in SUM_CASES])
def test_sum_order_contract_at_every_plan_branch(case):
    from bipymc_b200 import DeMcMpi, targets
    k, d, M, batches, prior = SUM_CASES[case]
    data = allcol_data(M, k)
    lik = targets.CudaSumLikelihood(ALLCOL_TERM + (ALLCOL_PRIOR if prior else ""), d, data, prior=prior, fmad=False)
    big = max(batches)
    th = _thetas(big, d)
    out = np.zeros(big, dtype=bool)
    if prior:
        out[5::9] = True                        # several chains of every 64-chain tile are outside the prior
        th[out, 0] = 7.0
    s = _sampler(DeMcMpi, lik, np.full(d, 0.1), 64)
    full = _eval(s, th)
    head = 35
    for b in batches:
        if b == big:
            continue
        got = np.concatenate([_eval(s, th[i:i + b]) for i in range(0, head, b)])[:head]
        assert np.array_equal(got, full[:head], equal_nan=True), "batch %d" % b
    if prior:
        assert np.all(full[out] == -np.inf)
    assert np.all(np.isfinite(full[~out]))
    pick = np.unique(np.r_[np.arange(head), np.linspace(0, big - 1, 16 if M > 20000 else 64).astype(int)])
    pick = pick[~out[pick]]
    ref = np.array([sum_order(allcol_terms_np(th[i], data)) for i in pick])
    bad = np.flatnonzero(full[pick] != ref)
    assert bad.size == 0, "rows %r: device %r, order contract %r" % (pick[bad][:4], full[pick][bad][:4], ref[bad][:4])


# ---- B. against the correctly rounded sum ---------------------------------------------------------------------
@pytest.mark.parametrize("M", [3000, 100003])
def test_sum_within_tree_bound_of_exact_sum(M):
    """LIN_TERM with the default fmad=True.  Error bound, with u = 2^-53 and A = sum_i (|theta0 x_i0| + |theta1 x_i1|):
      * each term t_i = theta0 x_i0 - theta1 x_i1 is made with at most two roundings (two products and a difference,
        or one product and a fused multiply-add), so |t^_i - t_i| <= (2u + u^2)(|theta0 x_i0| + |theta1 x_i1|);
      * the device adds the t^_i (and exact 0.0 pads) in a binary tree: 8 levels inside a chunk of 256 rows, then
        D_c = ceil(log2 chunks) levels over the chunk partials.  Every t^_i passes through at most D = 8 + D_c
        rounded adds, so |S^ - sum t^_i| <= gamma_D sum |t^_i|, gamma_D = D u / (1 - D u) (Higham, ch. 4);
      * sum |t^_i| <= (1 + 3u) A.
    Together: |S^ - S| <= (gamma_D (1 + 3u) + 2u + u^2) A.  A is itself summed in float64 (relative error below
    M u), so it is taken with a factor 1 + 1e-9."""
    from bipymc_b200 import DeMcMpi, targets
    k, d = 2, 2
    data = allcol_data(M, k, seed=3)
    s = _sampler(DeMcMpi, targets.CudaSumLikelihood(LIN_TERM, d, data), np.full(d, 0.1), 64)
    th = _thetas(4096, d, seed=4)
    got = _eval(s, th)
    nch = -(-M // CHUNK)
    D = 8 + (nch - 1).bit_length()
    gamma = D * U / (1.0 - D * U)
    for i in range(0, 4096, 256):
        exact = lin_exact_sum(th[i], data)
        A = np.sum(np.abs(th[i, 0] * data[:, 0]) + np.abs(th[i, 1] * data[:, 1])) * (1.0 + 1e-9)
        bound = (gamma * (1.0 + 3.0 * U) + 2.0 * U + U * U) * A
        assert abs(got[i] - exact) <= bound, (i, got[i], exact, abs(got[i] - exact) / bound)
        # the bound is tight enough to see one chunk of 256 rows dropped or counted twice
        chunks = [lin_exact_sum(th[i], data[j:j + CHUNK]) for j in range(0, M, CHUNK)]
        assert min(abs(c) for c in chunks) > 2.0 * bound, (i, min(abs(c) for c in chunks), bound)


# ---- C. user likelihoods in the generic kernels against the oracle step -----------------------------------------
def gauss_diag_np(theta, data):
    """GAUSS_DIAG for rows theta[n, d], the same operations in the same order (fmad=False)."""
    theta = np.atleast_2d(theta)
    d = theta.shape[1]
    s = np.zeros(theta.shape[0])
    for q in range(d):
        r = (theta[:, q] - data[q]) * data[d + q]
        s = s + r * r
    return -0.5 * s


ALGOS = {"dream_ncr3": ("dream", 3), "dream_ncr6": ("dream", 6), "demc": ("demc", None)}


def _algo(name, **dream_kw):
    from bipymc_b200 import DeMcMpi, DreamMpi
    algo, n_cr = ALGOS[name]
    if algo == "demc":
        return DeMcMpi, {}
    return DreamMpi, dict(n_cr=n_cr, **dream_kw)


def _oracle_run(s, oracle, algo):
    """The oracle step of test_native_gpu.py, with the split kernels (never the fused half-phase) shown to run."""
    from bipymc_b200 import _lib
    _lib.check(s._libh.bpm_profile(s._handle, 1))
    gens = 5
    if algo == "demc":
        _native_vs_oracle(s, oracle, gens=gens, k0=5, run_kwargs=dict(epsilon=1e-9))
    else:
        _native_vs_oracle(s, oracle, gens=gens, k0=2)
    k = launches_by_kind(s)
    _lib.check(s._libh.bpm_profile(s._handle, 0))
    assert k["fused_phase"] == 0 and k["propose"] == k["likelihood"] == k["accept"] == 2 * gens, k


@pytest.mark.parametrize("algo", sorted(ALGOS))
@pytest.mark.parametrize("d", ORACLE_DIMS)
def test_cuda_likelihood_generic_kernels_match_oracle(d, algo):
    from bipymc_b200 import targets
    data = gauss_diag_data(d)
    cls, kw = _algo(algo, n_cr_gen=2, burnin_gen=1000)
    np.random.seed(7)
    s = cls(_never, data[:d] + 0.2, n_chains=40 if d > 32 else 24, seed=31, varepsilon=0.3, fused=1,
            ln_like_cuda=targets.CudaLikelihood(GAUSS_DIAG, d, data, fmad=False), **kw)
    _oracle_run(s, lambda th: gauss_diag_np(th, data)[0], ALGOS[algo][0])


@pytest.mark.parametrize("algo", sorted(ALGOS))
@pytest.mark.parametrize("d,k,M", ORACLE_SUM)
def test_cuda_sum_likelihood_generic_kernels_match_oracle(d, k, M, algo):
    from bipymc_b200 import targets
    data = allcol_data(M, k)
    cls, kw = _algo(algo, n_cr_gen=2, burnin_gen=1000)
    np.random.seed(8)
    s = cls(_never, np.full(d, 0.05), n_chains=24, seed=32, varepsilon=0.02, fused=1,
            ln_like_cuda=targets.CudaSumLikelihood(ALLCOL_TERM, d, data, fmad=False), **kw)
    _oracle_run(s, lambda th: sum_order(allcol_terms_np(th, data)), ALGOS[algo][0])


# ---- D. the multi-problem contract at the untested shapes -------------------------------------------------------
G_D = 20


def _problem_set(n, d):
    return np.stack([gauss_diag_data(d, seed=g) for g in range(n_problems(n))])


def _contract_run(n, d, algo):
    cls, kw = _algo(algo, n_cr_gen=2, burnin_gen=G_D - 3)     # CR adaptation from generation 2 to 17 of 20
    ms = _multi(cls, GAUSS_DIAG, d, _problem_set(n, d), np.zeros(d), n, varepsilon=0.3, fused=1, **kw)
    singles = [_single_like(ms, cls, GAUSS_DIAG, d, g, fused=1, **kw) for g in range(ms.n_problems)]
    ms.run_mcmc(n * (G_D + 1))
    assert ms._hist.length == G_D + 1 and np.all(ms.n_accepted > 0)
    for g, s in enumerate(singles):
        s.run_mcmc(n * (G_D + 1))
        _assert_problem_equal(ms, g, s, ALGOS[algo][0] == "dream")
    if ALGOS[algo][0] == "dream":
        assert np.all(ms.n_cr_updates.sum(axis=1) > 0)
    return ms, singles


@pytest.mark.parametrize("algo", sorted(ALGOS))
@pytest.mark.parametrize("d", D_DIMS)
@pytest.mark.parametrize("n", D_CHAINS)
def test_each_problem_equals_its_single_problem_sampler(n, d, algo):
    _contract_run(n, d, algo)


def test_single_problem_sampler_of_a_set_matches_oracle():
    """Ties the multi-problem path to the oracle: problem 1 of a set equals its single-problem sampler, and that
    sampler's next generations equal the oracle step."""
    n, d, algo = 129, 20, "dream_ncr6"
    ms, singles = _contract_run(n, d, algo)
    data = ms._ln_like_cuda.data[1]
    _oracle_run(singles[1], lambda th: gauss_diag_np(th, data)[0], "dream")


@pytest.mark.parametrize("d", D_DIMS)
def test_problem_set_eval_matches_numpy_per_problem(d):
    """bpm_eval_lnl on a multi-problem handle (lnl_jit_problems_kernel): rows [g r, (g + 1) r) use data row g."""
    from bipymc_b200 import DeMcMpi
    data = _problem_set(129, d)
    P, r = data.shape[0], 1000
    ms = _multi(DeMcMpi, GAUSS_DIAG, d, data, np.zeros(d), 129, varepsilon=0.3)
    th = np.random.RandomState(d).uniform(-2.0, 2.0, (P * r, d))
    got = _eval(ms, th)
    for g in range(P):
        assert np.array_equal(got[g * r:(g + 1) * r], gauss_diag_np(th[g * r:(g + 1) * r], data[g])), g
