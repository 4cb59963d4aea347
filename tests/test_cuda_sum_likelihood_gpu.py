"""Per-observation CUDA likelihoods (targets.CudaSumLikelihood) on the GPU.

  * the order contract: the device sum equals the numpy restatement bit for bit, whatever the batch
    size or the number of chains;
  * a run's cached ln L equals bpm_eval_lnl of its final states;
  * agreement with the whole-function CudaLikelihood of the same model;
  * which kernels ran (never the fused half-phase);
  * RNG-replay parity with the reference's golden history;
  * the analytic posterior of a linear-Gaussian model;
  * the box prior, NaN, and a million observations."""
import numpy as np
import pytest

from test_cuda_sum_likelihood_cpu import (CHUNK, EXPFIT_PRIOR, EXPFIT_TERM, LINEFIT_PRIOR, LINEFIT_TERM, POLY_TERM,
                                          expfit_rows, linefit_rows, poly_data, poly_terms_np, sum_order)
from test_replay_parity_gpu import ALL_CASES, check_against_reference, launches_by_kind, oracle_traces

pytestmark = pytest.mark.gpu


def _never(theta, **kw):
    raise AssertionError("ln_like_fn must not be called when ln_like_cuda is given")


def _sampler(cls, lik, theta0, N, seed=11, **kw):
    np.random.seed(5)
    return cls(_never, np.asarray(theta0, dtype=float), n_chains=N, seed=seed, ln_like_cuda=lik, **kw)


def _eval(s, theta):
    """bpm_eval_lnl of host rows theta[n, d] on sampler s."""
    import torch
    rows = torch.zeros((theta.shape[0], s._ld), dtype=torch.float64, device=s._device)
    rows[:, :s.dim] = torch.from_numpy(np.ascontiguousarray(theta)).to(s._device)
    out = s._eval_lnl_rows(rows)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _thetas(n, d, seed=3):
    rs = np.random.RandomState(seed)
    return np.arange(1, d + 1) * 0.3 + 0.01 * rs.randn(n, d)


@pytest.mark.parametrize("M", [1, 31, CHUNK - 1, CHUNK, CHUNK + 1, 100003])
def test_order_contract_bit_for_bit(M):
    from bipymc_b200 import DeMcMpi, targets
    d = 3
    data = poly_data(M, d)
    lik = targets.CudaSumLikelihood(POLY_TERM, d, data, fmad=False)
    th = _thetas(4096, d)
    small = _sampler(DeMcMpi, lik, th[0], 64)
    got = {b: np.concatenate([_eval(small, th[i:i + b]) for i in range(0, 4096, b)]) for b in (1, 7, 4096)}
    assert np.array_equal(got[1], got[4096]) and np.array_equal(got[7], got[4096])
    pick = np.arange(0, 4096, 1 if M < 1000 else 64)
    ref = np.array([sum_order(poly_terms_np(th[i], data)) for i in pick])
    assert np.array_equal(got[4096][pick], ref)
    big = _sampler(DeMcMpi, lik, th[0], 100000)          # 10^5 rows in one call: another launch shape
    assert np.array_equal(_eval(big, np.tile(th, (25, 1))[:100000]), np.tile(got[4096], 25)[:100000])


WHOLE_POLY = r'''
__device__ double ln_like(const double* theta, const double* data) {
  double s = 0.0;
  for (int i = 0; i < BPM_NDATA / 3; ++i) {
    const double* row = data + 3 * i;
    double model = theta[BPM_DIM - 1];
    for (int q = BPM_DIM - 2; q >= 0; --q) model = model * row[0] + theta[q];
    const double r = (row[1] - model) / row[2];
    s += -0.5 * (r * r);
  }
  return s;
}
'''


@pytest.mark.parametrize("d", [3, 5])
@pytest.mark.parametrize("M", [60, 100000])
def test_agrees_with_whole_function_form(M, d):
    from bipymc_b200 import DeMcMpi, targets
    data = poly_data(M, d)
    th = _thetas(512, d)
    s_sum = _sampler(DeMcMpi, targets.CudaSumLikelihood(POLY_TERM, d, data), th[0], 64)
    s_one = _sampler(DeMcMpi, targets.CudaLikelihood(WHOLE_POLY, d, data.ravel()), th[0], 64)
    a, b = _eval(s_sum, th), _eval(s_one, th)
    np.testing.assert_allclose(a, b, rtol=1e-12, atol=0)


@pytest.mark.parametrize("d", [3, 5])
def test_launches_never_fused(d):
    from bipymc_b200 import DreamMpi, _lib, targets
    data = poly_data(500, d)
    s = _sampler(DreamMpi, targets.CudaSumLikelihood(POLY_TERM, d, data), np.arange(1, d + 1) * 0.3, 1000,
                 varepsilon=1e-3, n_cr_gen=3, burnin_gen=1000, fused=1)
    _lib.check(s._libh.bpm_profile(s._handle, 1))
    G = 10
    s.run_mcmc(1000 * (G + 1))
    k = launches_by_kind(s)
    assert k["propose"] == k["likelihood"] == k["accept"] == 2 * G and k["fused_phase"] == 0, k


def test_replay_parity_linefit_dream():
    from bipymc_b200 import DreamMpi, targets
    name = "linefit_dream"
    case = ALL_CASES[name]
    osampler, traces = oracle_traces(name)
    lik = targets.CudaSumLikelihood(LINEFIT_TERM + LINEFIT_PRIOR, 3, linefit_rows(), prior=True, fmad=False)
    np.random.seed(case["seed"])
    s = DreamMpi(_never, np.asarray(case["theta_0"], dtype=float), n_chains=case["n_chains"], ln_like_cuda=lik,
                 **case["ctor_kwargs"])
    sink = []
    s.run_mcmc(case["n"], _replay=traces, _trace=sink, **case["run_kwargs"])
    check_against_reference(name, s, sink, traces, osampler)


LINE_BOX = POLY_TERM + r'''
__device__ double ln_prior(const double* theta) {
  return (fabs(theta[0]) < 100.0 && fabs(theta[1]) < 100.0) ? 0.0 : -INFINITY;
}
'''


def test_analytic_linear_gaussian_posterior():
    from bipymc_b200 import DreamMpi, targets
    M, N = 10000, 1024
    rs = np.random.RandomState(11)
    x = rs.uniform(0.0, 2.0, M)                          # correlated intercept and slope
    err = 0.05 + 0.1 * rs.rand(M)
    data = np.stack([x, 0.3 + 0.6 * x + err * rs.randn(M), err], axis=1)
    X = np.stack([np.ones(M), x], axis=1)
    W = 1.0 / err ** 2
    cov = np.linalg.inv(X.T @ (W[:, None] * X))
    mean = cov @ (X.T @ (W * data[:, 1]))
    sd = np.sqrt(np.diag(cov))
    lik = targets.CudaSumLikelihood(LINE_BOX, 2, data, prior=True)
    s = _sampler(DreamMpi, lik, mean + 2 * sd, N, varepsilon=(2 * sd) ** 2, n_cr_gen=5, burnin_gen=200)
    G = 600
    s.run_mcmc(N * (G + 1))
    h = s._hist.tensor()[G // 2:, :, :2].cpu().numpy().reshape(-1, 2)
    assert np.all(np.abs(h.mean(axis=0) - mean) < 0.1 * sd), (h.mean(axis=0), mean, sd)
    np.testing.assert_allclose(np.cov(h.T), cov, rtol=0.1)


HALF_PLANE = r'''
__device__ double ln_prior(const double* t) { return t[0] < 0.0 ? -INFINITY : 0.0; }
__device__ double ln_like_term(const double* t, const double* row) {
  return -0.5 * ((t[0] - row[0]) * (t[0] - row[0]) + t[1] * t[1]) / BPM_NROWS;
}
'''


@pytest.mark.parametrize("d", [2, 6])
def test_box_prior_is_never_left(d):
    from bipymc_b200 import DreamMpi, targets
    lik = targets.CudaSumLikelihood(HALF_PLANE, d, np.full(300, 0.2), prior=True)
    s = _sampler(DreamMpi, lik, np.r_[0.5, np.zeros(d - 1)], 1000, varepsilon=1e-2, n_cr_gen=3, burnin_gen=1000)
    s.run_mcmc(1000 * 31)
    h = s._hist.tensor()[:, :, :d].cpu().numpy()
    assert (h[:, :, 0] >= 0.0).all()
    assert np.isfinite(s._lnl.cpu().numpy()).all()
    assert 0 < s.n_accepted < s.n_accepted + s.n_rejected


def test_nan_raises():
    from bipymc_b200 import DeMcMpi, targets
    src = "__device__ double ln_like_term(const double* t, const double* r) { return t[0] > 1e300 ? 0.0 : NAN; }\n"
    s = _sampler(DeMcMpi, targets.CudaSumLikelihood(src, 2, np.ones(1000)), np.zeros(2), 64)
    with pytest.raises(ValueError, match="probabilities contain NaN"):
        s.run_mcmc(64 * 4)


def test_a_million_observations():
    from bipymc_b200 import DreamMpi, targets
    lik = targets.CudaSumLikelihood(EXPFIT_TERM + EXPFIT_PRIOR, 5, expfit_rows(1000000), prior=True)
    s = _sampler(DreamMpi, lik, [12.0, 1.5, 0.6, 1e-3, 2e-3], 256,
                 varepsilon=np.asarray([1e-2, 1e-2, 1e-3, 1e-8, 1e-9]) * 1e-2, n_cr_gen=3, burnin_gen=1000)
    s.run_mcmc(256 * 6)
    lnl = s._lnl.cpu().numpy()
    assert np.isfinite(lnl).all()
    assert np.array_equal(lnl, _eval(s, s._X[:, :5].cpu().numpy()))


def test_serial_demc_runs_the_sum_kernels():
    from bipymc_b200 import DeMc, targets
    data = poly_data(2000, 3)
    np.random.seed(2)
    s = DeMc(_never, n_chains=64, seed=3, ln_like_cuda=targets.CudaSumLikelihood(POLY_TERM, 3, data))
    s.run_mcmc(64 * 6, np.arange(1, 4) * 0.3, varepsilon=1e-4)
    lnl = s._lnl.cpu().numpy()
    assert np.isfinite(lnl).all()
    assert np.array_equal(lnl, _eval(s, s._X[:, :3].cpu().numpy()))


def test_dimension_mismatch_is_refused():
    from bipymc_b200 import DeMcMpi, targets
    with pytest.raises(ValueError, match="dimension"):
        DeMcMpi(_never, np.zeros(2), n_chains=64, ln_like_cuda=targets.CudaSumLikelihood(LINEFIT_TERM, 3, np.ones(9)))
