"""Per-observation likelihoods for many datasets in one sampler (targets.CudaSumLikelihoodSet) on the GPU.

  * the order contract: bpm_eval_lnl of problem g's rows equals the numpy restatement of the summation order over
    problem g's terms bit for bit, and a CudaSumLikelihood holding data[g], whatever the batch per problem;
  * the per-problem contract: problem g of a run equals a single-problem CudaSumLikelihood sampler with n chains,
    data[g], key problem_seeds[g] and the same initial states, bit for bit (history, cached ln L, CR state,
    counters), for DREAM and DE-MC, odd and even n, d = 3 and 5, with and without a prior, and with M large
    enough that the sum is split over several groups of chunks;
  * launches per generation do not depend on P, and the fused half-phase never runs;
  * no cross-talk: 1000 linear-Gaussian problems each match their own analytic posterior;
  * -inf and NaN in one problem, checkpoints, and the target shape (few chains, a million rows)."""
import numpy as np
import pytest

from test_cuda_sum_likelihood_cpu import (CHUNK, EXPFIT_PRIOR, EXPFIT_TERM, LINEFIT_PRIOR, LINEFIT_TERM, POLY_TERM,
                                          expfit_rows, linefit_rows, poly_data, poly_terms_np, sum_order)
from test_replay_parity_gpu import launches_by_kind

pytestmark = pytest.mark.gpu

P = 7
LINEFIT_THETA0 = [-0.9, 4.3, -0.7]
EXPFIT_THETA0 = [12.0, 1.5, 0.6, 1e-3, 2e-3]


def _never(theta, **kw):
    raise AssertionError("ln_like_fn must not be called when ln_like_cuda is given")


def _multi(cls, src, dim, data, theta0, n, prior=False, seed=11, varepsilon=1e-4, **kw):
    from bipymc_b200 import targets
    np.random.seed(5)
    lik = targets.CudaSumLikelihoodSet(src, dim, data, prior=prior, fmad=False)
    return cls(_never, np.asarray(theta0, dtype=float), n_chains=n, seed=seed, ln_like_cuda=lik,
               varepsilon=varepsilon, **kw)


def _single_like(ms, cls, g, **kw):
    """Problem g of multi-problem sampler ms as a CudaSumLikelihood sampler of its own, from the same states."""
    from bipymc_b200 import targets
    n, dim, lik = ms.n_chains, ms.dim, ms._ln_like_cuda
    one = targets.CudaSumLikelihood(lik.source, dim, lik.data[g], prior=lik.prior, fmad=lik.fmad)
    s = cls(_never, np.zeros(dim), n_chains=n, seed=ms.problem_seeds[g], ln_like_cuda=one, **kw)
    s.load_history(ms._hist.tensor()[:1, g * n:(g + 1) * n, :dim].cpu().numpy())
    return s


def _assert_problem_equal(ms, g, s, dream):
    n, d = ms.n_chains, ms.dim
    hm = ms._hist.tensor()[:, g * n:(g + 1) * n, :d].cpu().numpy()
    hs = s._hist.tensor()[:, :, :d].cpu().numpy()
    assert hm.shape == hs.shape
    np.testing.assert_array_equal(hm, hs, err_msg="history of problem %d" % g)
    np.testing.assert_array_equal(ms._lnl[g * n:(g + 1) * n].cpu().numpy(), s._lnl.cpu().numpy())
    assert ms.n_accepted[g] == s.n_accepted and ms.n_rejected[g] == s.n_rejected, (g, ms.n_accepted[g], s.n_accepted)
    np.testing.assert_array_equal(ms.acceptance_fraction[g], s.acceptance_fraction)
    if dream:
        np.testing.assert_array_equal(ms.p_cr[g], s.p_cr)
        np.testing.assert_array_equal(ms.delta_m[g], s.delta_m)
        np.testing.assert_array_equal(ms.n_cr_updates[g], s.n_cr_updates)


def _eval(s, theta):
    """bpm_eval_lnl of host rows theta[n, d] on sampler s (multi-problem: rows problem-major, n / P each)."""
    import torch
    rows = torch.zeros((theta.shape[0], s._ld), dtype=torch.float64, device=s._device)
    rows[:, :s.dim] = torch.from_numpy(np.ascontiguousarray(theta)).to(s._device)
    out = s._eval_lnl_rows(rows)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _poly_set(n_prob, M, d):
    return np.stack([poly_data(M, d, seed=7 + g) for g in range(n_prob)])


def _linefit_set(n_prob, seed=0):
    """The reference's line-fit rows with the ordinate shifted and rescaled per problem."""
    base = linefit_rows()
    rs = np.random.RandomState(seed)
    out = np.repeat(base[None], n_prob, axis=0)
    out[:, :, 1] = out[:, :, 1] * (1.0 + 0.05 * rs.randn(n_prob, 1)) + 0.2 * rs.randn(n_prob, 1)
    return out


def _expfit_set(n_prob, M=60, seed=0):
    base = expfit_rows(M)
    rs = np.random.RandomState(seed)
    out = np.repeat(base[None], n_prob, axis=0)
    out[:, :, 1] += 0.01 * rs.randn(n_prob, 1)
    return out


@pytest.mark.parametrize("M", [1, 31, CHUNK - 1, CHUNK, CHUNK + 1, 100003])
def test_order_contract_bit_for_bit(M):
    from bipymc_b200 import DeMcMpi, targets
    d, n_prob = 3, 3
    data = _poly_set(n_prob, M, d)
    ms = _multi(DeMcMpi, POLY_TERM, d, data, np.arange(1, d + 1) * 0.3, 8)
    rs = np.random.RandomState(3)
    B = 1024                                                  # rows per problem of the largest batch
    th = np.arange(1, d + 1) * 0.3 + 0.01 * rs.randn(n_prob, B, d)
    got = {b: np.concatenate([_eval(ms, th[:, i:i + b].reshape(-1, d)).reshape(n_prob, -1)
                              for i in range(0, B, b)], axis=1) for b in (1, 7, B)}
    assert np.array_equal(got[1], got[B]) and np.array_equal(got[7], got[B])
    pick = np.arange(0, B, 1 if M < 1000 else 128)
    for g in range(n_prob):
        ref = np.array([sum_order(poly_terms_np(th[g, i], data[g])) for i in pick])
        assert np.array_equal(got[B][g, pick], ref), g
        one = DeMcMpi(_never, th[g, 0], n_chains=8, seed=1,
                      ln_like_cuda=targets.CudaSumLikelihood(POLY_TERM, d, data[g], fmad=False))
        assert np.array_equal(_eval(one, th[g]), got[B][g]), g


# name: (term, prior source, dim, data(P), theta0, varepsilon)
CASES = {"poly_d3": (POLY_TERM, None, 3, lambda p: _poly_set(p, 60, 3), [0.3, 0.6, 0.9], 1e-4),
         "linefit_prior_d3": (LINEFIT_TERM, LINEFIT_PRIOR, 3, _linefit_set, LINEFIT_THETA0, 1e-3),
         "expfit_prior_d5": (EXPFIT_TERM, EXPFIT_PRIOR, 5, _expfit_set, EXPFIT_THETA0, 1e-8),
         "poly_d5_groups": (POLY_TERM, None, 5, lambda p: _poly_set(p, 3000, 5), [0.3, 0.6, 0.9, 1.2, 1.5], 1e-6)}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("n", [33, 64])
@pytest.mark.parametrize("algo", ["dream", "demc"])
def test_each_problem_equals_its_single_problem_sampler(case, n, algo):
    from bipymc_b200 import DeMcMpi, DreamMpi
    term, prior_src, dim, data_fn, theta0, var = CASES[case]
    cls = DreamMpi if algo == "dream" else DeMcMpi
    # CR adaptation switches on after 3 rows and off at generation 14; gamma jumps every 5 / 10 generations
    kw = dict(n_cr_gen=3, burnin_gen=14) if algo == "dream" else {}
    ms = _multi(cls, term + (prior_src or ""), dim, data_fn(P), theta0, n, prior=prior_src is not None,
                varepsilon=var, **kw)
    singles = [_single_like(ms, cls, g, **kw) for g in range(P)]
    G = 26
    ms.run_mcmc(n * (G + 1))
    assert ms._hist.length == G + 1
    assert np.all(ms.n_accepted > 0)
    for g, s in enumerate(singles):
        s.run_mcmc(n * (G + 1))
        _assert_problem_equal(ms, g, s, algo == "dream")
    h = ms._hist.tensor()[-1, :, :dim].cpu().numpy()
    assert not np.array_equal(h[:n], h[n:2 * n])               # the problems differ: their data do


@pytest.mark.parametrize("d", [3, 5])
def test_launches_per_generation_do_not_depend_on_p(d):
    from bipymc_b200 import DreamMpi, _lib
    G = 8
    counts = []
    for n_prob in (P, 1000):
        ms = _multi(DreamMpi, POLY_TERM, d, _poly_set(n_prob, 500, d), np.arange(1, d + 1) * 0.3, 32,
                    n_cr_gen=3, burnin_gen=100)
        _lib.check(ms._libh.bpm_profile(ms._handle, 1))
        ms.run_mcmc(32 * (G + 1))
        counts.append(launches_by_kind(ms))
    assert counts[0] == counts[1], counts
    k = counts[0]
    assert k["split"] == G and k["cr_reduce"] == G, k
    assert k["fused_phase"] == 0 and k["propose"] == k["likelihood"] == k["accept"] == 2 * G, k


def test_no_cross_talk_at_scale():
    """1000 problems x 64 chains, y = a_g + b_g x + N(0, sigma^2) with known sigma, 300 rows each: every problem's
    posterior is Gaussian with its own mean and covariance (flat prior)."""
    from bipymc_b200 import DreamMpi
    n_prob, n, M = 1000, 64, 300
    rs = np.random.RandomState(7)
    x = np.linspace(-1.0, 1.0, M)
    a, b = rs.uniform(-5, 5, n_prob), rs.uniform(-3, 3, n_prob)
    sig = 0.3 + 0.2 * rs.rand(n_prob, M)
    y = a[:, None] + b[:, None] * x[None] + sig * rs.randn(n_prob, M)
    data = np.stack([np.broadcast_to(x, (n_prob, M)), y, sig], axis=2)      # rows (x, y, sigma): POLY_TERM at d = 2
    X = np.stack([np.ones(M), x], axis=1)
    mean, sd = np.zeros((n_prob, 2)), np.zeros((n_prob, 2))
    for g in range(n_prob):
        W = 1.0 / sig[g] ** 2
        cov = np.linalg.inv(X.T @ (W[:, None] * X))
        mean[g] = cov @ (X.T @ (W * y[g]))
        sd[g] = np.sqrt(np.diag(cov))
    ms = _multi(DreamMpi, POLY_TERM, 2, data, mean, n, varepsilon=1e-3, n_cr_gen=5, burnin_gen=200)
    G = 400
    ms.run_mcmc(n * (G + 1))
    m, s, _ = ms.param_est(n * (G // 2))
    assert m.shape == s.shape == (n_prob, 2)
    z = np.abs(m - mean) / sd
    assert z.max() < 0.35, (z.max(), np.unravel_index(z.argmax(), z.shape))
    np.testing.assert_allclose(s, sd, rtol=0.2)
    assert ms.rhat().shape == (n_prob, 2) and np.all(ms.rhat() < 1.2)
    acc = ms.acceptance_fraction
    assert acc.shape == (n_prob,) and np.all((acc > 0.05) & (acc < 0.95))
    assert ms.p_cr.shape == (n_prob, 3)
    assert ms.super_chain.shape == (n_prob, n * (G + 1), 2)


# row = (bound, nan flag): -inf above a problem-specific bound, NaN where the data say so
BOUNDED = r'''
__device__ double ln_prior(const double* t) { return fabs(t[1]) < 1e3 ? 0.0 : -INFINITY; }
__device__ double ln_like_term(const double* t, const double* row) {
  if (t[0] > row[0]) return -INFINITY;
  if (row[1] != 0.0) return NAN;
  return -0.5 * (t[0] * t[0] + t[1] * t[1]) / BPM_NROWS;
}
'''


def test_minus_inf_stays_in_its_problem():
    from bipymc_b200 import DreamMpi
    data = np.zeros((P, 300, 2))
    data[:, :, 0] = 100.0
    data[3, 150, 0] = 0.0                  # one row of problem 3 bounds t[0] <= 0
    ms = _multi(DreamMpi, BOUNDED, 2, data, [-0.5, 0.0], 32, prior=True, varepsilon=1e-2)
    ms.run_mcmc(32 * 61)
    h = ms._hist.tensor()[:, :, :2].cpu().numpy().reshape(-1, P, 32, 2)
    assert (h[:, 3, :, 0] <= 0.0).all()
    assert all((h[:, g, :, 0] > 0.0).any() for g in range(P) if g != 3)
    assert np.isfinite(ms._lnl.cpu().numpy()).all()


def test_nan_in_one_problem_raises():
    from bipymc_b200 import DeMcMpi
    data = np.zeros((P, 300, 2))
    data[:, :, 0] = 100.0
    data[2, 299, 1] = 1.0
    ms = _multi(DeMcMpi, BOUNDED, 2, data, [-0.5, 0.0], 32, prior=True, varepsilon=1e-2)
    with pytest.raises(ValueError, match="probabilities contain NaN"):
        ms.run_mcmc(32 * 4)


@pytest.mark.parametrize("ext", [".h5", ".npz"])
def test_checkpoint_resumes_bit_for_bit(tmp_path, ext):
    from bipymc_b200 import DreamMpi
    path = str(tmp_path / ("ck" + ext))
    kw = dict(n_cr_gen=3, burnin_gen=30)
    src = LINEFIT_TERM + LINEFIT_PRIOR
    a = _multi(DreamMpi, src, 3, _linefit_set(P), LINEFIT_THETA0, 33, prior=True, seed=[5, 9, 2, 7, 1, 3, 8],
               varepsilon=1e-3, **kw)
    a.run_mcmc(33 * 13)
    a.save_state(path)
    a.run_mcmc(33 * 13)
    b = _multi(DreamMpi, src, 3, _linefit_set(P), LINEFIT_THETA0, 33, prior=True, seed=0, varepsilon=1e-3, **kw)
    b.load_state(path)
    assert b.problem_seeds == [5, 9, 2, 7, 1, 3, 8]
    np.testing.assert_array_equal(b.p_cr.shape, (P, 3))
    b.run_mcmc(33 * 13)
    np.testing.assert_array_equal(a._hist.tensor()[:, :, :3].cpu().numpy(), b._hist.tensor()[:, :, :3].cpu().numpy())
    np.testing.assert_array_equal(a._lnl.cpu().numpy(), b._lnl.cpu().numpy())
    np.testing.assert_array_equal(a.p_cr, b.p_cr)
    np.testing.assert_array_equal(a.n_accepted, b.n_accepted)


def test_few_chains_a_million_rows():
    """The shape the sum set is for: P = 16 problems of 8 chains, 10^6 rows each."""
    from bipymc_b200 import DreamMpi
    n_prob, n = 16, 8
    ms = _multi(DreamMpi, EXPFIT_TERM + EXPFIT_PRIOR, 5, _expfit_set(n_prob, M=1000000), EXPFIT_THETA0, n,
                prior=True, varepsilon=np.asarray([1e-2, 1e-2, 1e-3, 1e-8, 1e-9]) * 1e-2, n_cr_gen=3, burnin_gen=1000)
    ms.run_mcmc(n * 6)
    lnl = ms._lnl.cpu().numpy()
    assert lnl.shape == (n_prob * n,) and np.isfinite(lnl).all()
    assert np.array_equal(lnl, _eval(ms, ms._X[:, :5].cpu().numpy()))
