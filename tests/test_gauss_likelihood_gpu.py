"""Gaussian likelihoods with a dense data covariance (targets.CudaGaussLikelihood) on the GPU.

  A. values against numpy within an error bound derived from M and the magnitudes, a bound tight enough to
     catch one dropped column block or observation;
  B. the same theta rows give the same bits at any batch size, chain count, tile size and slice;
  C. the prior: -inf wherever it is -inf (model_mean NaN there), else prior + the value without it, bit for bit;
  D. sampler steps against the oracle step, and proof that no fused half-phase ran; serial DE-MC;
  E. the analytic posterior of a linear model with exponential-kernel noise, which a diagonal fit misses;
  F. a refused bpm_set_jit_gauss_target changes nothing, and destroyed handles release their memory."""
import ctypes as C

import numpy as np
import pytest

from test_gauss_likelihood_cpu import (A_CASES, ALLCOL_MEAN, D_CASES, HALF_PLANE_MEAN, HALF_PLANE_PRIOR, LINEAR_MEAN,
                                       allcol_mean_np, case_data, exp_cov, gauss_lnl_np, half_plane_prior_np)
from test_jit_shapes_gpu import ALGOS, _algo, _oracle_run

pytestmark = pytest.mark.gpu

U = 2.0 ** -53          # unit roundoff of float64


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


def _gamma(n):
    return n * U / (1.0 - n * U)


def error_bound(mean, y, B, c0):
    """|device - numpy| bound per row.  Both compute z_j = sum_k r_k B_kj, r = mean - y (the same rounded r), in
    different orders: each is within gamma_M a_j of the exact z_j, a_j = sum_k |r_k B_kj|.  The squares' sum adds
    M non-negative terms, within gamma_(M+1) of its exact value in any order; then c0 + maha and the half."""
    M = y.size
    r = np.atleast_2d(mean) - y[None, :]
    z = r @ B
    a = np.abs(r) @ np.abs(B)
    g = _gamma(M)
    dz = 2.0 * g * a * (1.0 + 1e-6)
    maha = np.sum(z * z, axis=1)
    dmaha = np.sum(dz * (2.0 * np.abs(z) + dz), axis=1) + 2.0 * _gamma(M + 1) * maha
    return 0.5 * dmaha + 4.0 * U * (abs(c0) + maha) + 1e-300


# ---- A. values ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,d,k", A_CASES)
def test_values_within_the_derived_bound(M, d, k):
    from bipymc_b200 import DeMcMpi, targets
    x, y, cov, theta0 = case_data(M, d, k)
    lik = targets.CudaGaussLikelihood(ALLCOL_MEAN, d, x, y, cov, fmad=False)
    th = theta0 + 0.02 * np.random.RandomState(M + d).randn(300, d)
    s = _sampler(DeMcMpi, lik, theta0, 64)
    got = _eval(s, th)
    mean = allcol_mean_np(th, x)
    ref = gauss_lnl_np(mean, y, lik.B, lik.c0)
    bound = error_bound(mean, y, lik.B, lik.c0)
    err = np.abs(got - ref)
    assert np.all(err <= bound), (err.max(), bound[np.argmax(err / bound)])
    # the bound is tight enough to see the last column block, or the first observation, go missing
    Bc = lik.B.copy()
    Bc[:, 128 * ((M - 1) // 128):] = 0.0
    assert np.all(np.abs(gauss_lnl_np(mean, y, Bc, lik.c0) - ref) > bound)
    mo = mean.copy()
    mo[:, 0] = y[0]
    assert np.mean(np.abs(gauss_lnl_np(mo, y, lik.B, lik.c0) - ref) > bound) >= 0.9


# ---- B. batch independence ------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [1000, 4096])
def test_bits_do_not_depend_on_the_batch(M):
    from bipymc_b200 import DeMcMpi, targets
    d, k = 5, 3
    x, y, cov, theta0 = case_data(M, d, k)
    lik = targets.CudaGaussLikelihood(ALLCOL_MEAN, d, x, y, cov, fmad=False)
    n = 20000 if M == 1000 else 70000          # 20000 rows take 64-row tiles; 70000 at M = 4096 run in two slices
    th = theta0 + 0.02 * np.random.RandomState(1).randn(n, d)
    small = _sampler(DeMcMpi, lik, theta0, 64)
    full = _eval(small, th)
    assert np.all(np.isfinite(full))
    by4096 = np.concatenate([_eval(small, th[i:i + 4096]) for i in range(0, n, 4096)])
    assert np.array_equal(by4096, full)
    by7 = np.concatenate([_eval(small, th[i:i + 7]) for i in range(0, 700, 7)])
    assert np.array_equal(by7, full[:700])
    by1 = np.concatenate([_eval(small, th[i:i + 1]) for i in range(64)])
    assert np.array_equal(by1, full[:64])
    big = _sampler(DeMcMpi, lik, theta0, 1000)
    assert np.array_equal(_eval(big, th[:4096]), full[:4096])


# ---- C. the prior --------------------------------------------------------------------------------------------
def test_prior_short_circuits_and_is_added_last():
    from bipymc_b200 import DeMcMpi, DreamMpi, targets
    M = 300
    x = np.random.RandomState(2).uniform(0.0, 1.0, M)
    cov = exp_cov(np.linspace(0.0, 1.0, M), 0.2, 0.1, 1e-4)
    y = 0.5 * x + 0.25 + np.linalg.cholesky(cov) @ np.random.RandomState(3).randn(M)
    with_p = targets.CudaGaussLikelihood(HALF_PLANE_MEAN + HALF_PLANE_PRIOR, 2, x, y, cov, prior=True, fmad=False)
    without = targets.CudaGaussLikelihood(HALF_PLANE_MEAN, 2, x, y, cov, fmad=False)
    th = np.stack([np.random.RandomState(4).uniform(-0.5, 0.5, 2000), np.random.RandomState(5).uniform(0, 0.5, 2000)],
                  axis=1)
    a = _eval(_sampler(DeMcMpi, with_p, [0.25, 0.25], 64), th)
    b = _eval(_sampler(DeMcMpi, without, [0.25, 0.25], 64), th)
    neg = th[:, 0] < 0.0
    assert neg.sum() > 500 and np.all(np.isnan(b[neg]))
    assert np.all(a[neg] == -np.inf)
    assert np.array_equal(a[~neg], half_plane_prior_np(th[~neg]) + b[~neg])
    # a sampler that keeps proposing outside the prior never sees the NaN there: data with slope 0 put the
    # posterior of theta[0] at the boundary; every chain starts inside
    flat = targets.CudaGaussLikelihood(HALF_PLANE_MEAN + HALF_PLANE_PRIOR, 2, x, y - 0.5 * x, cov, prior=True,
                                       fmad=False)
    s = _sampler(DreamMpi, flat, [0.05, 0.25], 512, varepsilon=1e-5, n_cr_gen=3, burnin_gen=1000)
    assert np.isfinite(s._lnl.cpu().numpy()).all()
    s.run_mcmc(512 * 31)
    h = s._hist.tensor()[:, :, :2].cpu().numpy()
    assert (h[:, :, 0] >= 0.0).all() and np.isfinite(s._lnl.cpu().numpy()).all()
    assert 0 < s.n_accepted < s.n_accepted + s.n_rejected
    with_p_out = _eval(s, np.array([[-0.01, 0.25], [-1.0, 0.0]]))
    assert np.all(with_p_out == -np.inf)


# ---- D. sampler steps against the oracle ----------------------------------------------------------------------
@pytest.mark.parametrize("algo", sorted(ALGOS))
@pytest.mark.parametrize("d,M", D_CASES)
def test_sampler_steps_match_oracle(d, M, algo):
    from bipymc_b200 import targets
    k = 3
    x, y, cov, theta0 = case_data(M, d, k, seed=9)
    lik = targets.CudaGaussLikelihood(ALLCOL_MEAN, d, x, y, cov, fmad=False)
    cls, kw = _algo(algo, n_cr_gen=2, burnin_gen=1000)
    np.random.seed(8)
    s = cls(_never, theta0, n_chains=24, seed=32, varepsilon=1e-4, fused=1, ln_like_cuda=lik, **kw)
    _oracle_run(s, lambda t: gauss_lnl_np(allcol_mean_np(t, x), y, lik.B, lik.c0)[0], ALGOS[algo][0])


def test_serial_demc_runs_the_gauss_kernels():
    from bipymc_b200 import DeMc, targets
    x, y, cov, theta0 = case_data(500, 3, 2)
    lik = targets.CudaGaussLikelihood(ALLCOL_MEAN, 3, x, y, cov)
    np.random.seed(2)
    s = DeMc(_never, n_chains=64, seed=3, ln_like_cuda=lik)
    s.run_mcmc(64 * 6, theta0, varepsilon=1e-4)
    lnl = s._lnl.cpu().numpy()
    assert np.isfinite(lnl).all()
    assert np.array_equal(lnl, _eval(s, s._X[:, :3].cpu().numpy()))


# ---- E. statistics ---------------------------------------------------------------------------------------------
BOX_PRIOR = r'''
__device__ double ln_prior(const double* theta) {
  for (int q = 0; q < BPM_DIM; ++q) if (fabs(theta[q]) > 100.0) return -INFINITY;
  return 0.0;
}
'''
DIAG_TERM = r'''
__device__ double ln_like_term(const double* theta, const double* row) {   // row = (1, t, t^2, y, var)
  const double r = row[3] - (theta[0] * row[0] + theta[1] * row[1] + theta[2] * row[2]);
  return -0.5 * r * r / row[4];
}
'''


def test_analytic_posterior_of_a_linear_model_with_correlated_noise():
    from bipymc_b200 import DreamMpi, targets
    M, d, N, G = 512, 3, 512, 3000
    t = np.linspace(0.0, 1.0, M)
    A = np.stack([np.ones(M), t, t * t], axis=1)
    cov = exp_cov(t, 0.2, 0.1, 1e-4)
    y = A @ np.array([0.5, -1.0, 2.0]) + np.linalg.cholesky(cov) @ np.random.RandomState(21).randn(M)
    Ci = np.linalg.inv(cov)
    S = np.linalg.inv(A.T @ Ci @ A)
    mu = S @ (A.T @ Ci @ y)
    sd = np.sqrt(np.diag(S))
    lik = targets.CudaGaussLikelihood(LINEAR_MEAN + BOX_PRIOR, d, A, y, cov, prior=True)
    s = _sampler(DreamMpi, lik, mu + sd, N, varepsilon=(0.1 * sd) ** 2, n_cr_gen=5, burnin_gen=300)
    s.run_mcmc(N * (G + 1))
    h = s._hist.tensor()[G // 2:, :, :d].cpu().numpy()
    chain_means = h.mean(axis=0)                               # [N, d]
    mcse = chain_means.std(axis=0, ddof=1) / np.sqrt(N)
    flat = h.reshape(-1, d)
    assert np.all(np.abs(flat.mean(axis=0) - mu) < 4.0 * mcse), (flat.mean(axis=0), mu, mcse)
    corr = np.corrcoef(flat.T)
    assert np.all(np.abs(corr - S / np.outer(sd, sd)) < 0.03), (corr, S / np.outer(sd, sd))
    np.testing.assert_allclose(flat.std(axis=0), sd, rtol=0.1)
    # the diagonal-only per-observation fit of the same data: its posterior sd misses the analytic one by >= 2x
    rows = np.concatenate([A, y[:, None], np.diag(cov)[:, None]], axis=1)
    diag = targets.CudaSumLikelihood(DIAG_TERM + BOX_PRIOR, d, rows, prior=True)
    s2 = _sampler(DreamMpi, diag, mu + 0.1 * sd, N, varepsilon=(0.01 * sd) ** 2, n_cr_gen=5, burnin_gen=300)
    s2.run_mcmc(N * (G + 1))
    sd2 = s2._hist.tensor()[G // 2:, :, :d].cpu().numpy().reshape(-1, d).std(axis=0)
    assert np.all(sd / sd2 >= 2.0), (sd, sd2)


# ---- F. handle lifecycle ------------------------------------------------------------------------------------------
def test_refused_set_target_changes_nothing():
    import torch
    from bipymc_b200 import DreamMpi, _lib, targets
    x, y, cov, theta0 = case_data(200, 4, 2)
    lik = targets.CudaGaussLikelihood(ALLCOL_MEAN, 4, x, y, cov)
    out = []
    for refuse in (False, True):
        s = _sampler(DreamMpi, lik, theta0, 256, varepsilon=1e-4, n_cr_gen=2, burnin_gen=100)
        if refuse:
            lib, h = s._libh, s._handle
            bad = lik.B.copy()
            bad[5, 2] = 1e-3                                   # below the diagonal
            p = _lib.dptr
            log = C.create_string_buffer(4096)
            rc = lib.bpm_set_jit_gauss_target(h, lik.source.encode(), p(lik.data), 200, 2, p(lik.y), p(bad), lik.c0,
                                              1, None, log, 4096)
            assert rc != 0 and b"upper triangular" in lib.bpm_last_error()
            rc = lib.bpm_set_jit_gauss_target(h, b"__device__ double model_mean(const double* t, const double* r) {",
                                              p(lik.data), 200, 2, p(lik.y), p(lik.B), lik.c0, 1, None, log, 4096)
            assert rc != 0 and log.value
            assert lib.bpm_set_target(h, _lib.TARGET_JIT_GAUSS, None, 0) != 0
            assert b"bpm_set_jit_gauss_target" in lib.bpm_last_error()
        s.run_mcmc(256 * 6)
        torch.cuda.synchronize()
        out.append((s._X.cpu().numpy().copy(), s._lnl.cpu().numpy().copy()))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])


def test_multi_problem_handles_are_refused():
    from bipymc_b200 import _lib
    from test_handle_lifecycle_gpu import _create
    lib = _lib.load()
    h = _create(lib, 16, 2)
    try:
        _lib.check(lib.bpm_set_problems(h, 2, (C.c_uint64 * 2)(1, 2)))
        z = np.zeros(4)
        assert lib.bpm_set_jit_gauss_target(h, ALLCOL_MEAN.encode(), _lib.dptr(z), 4, 1, _lib.dptr(z),
                                            _lib.dptr(np.eye(4)), 1.0, 0, None, None, 0) != 0
        assert b"multi-problem" in lib.bpm_last_error()
    finally:
        lib.bpm_destroy(h)


def test_destroyed_handles_release_their_device_memory():
    import torch
    from bipymc_b200 import _lib, targets
    from test_handle_lifecycle_gpu import _Pop, _create
    lib = _lib.load()
    torch.cuda.set_device(0)
    M, d, n = 4096, 4, 512
    x, y, cov, theta0 = case_data(M, d, 1)
    lik = targets.CudaGaussLikelihood(ALLCOL_MEAN, d, x, y, cov)
    X0 = torch.from_numpy(theta0 + 0.01 * np.random.RandomState(0).randn(n, d)).to("cuda")
    pop = _Pop(n, d)

    def cycle():
        h = _create(lib, n, d)
        lik._attach(lib, h)
        st = pop.start(lib, h, X0)
        _lib.check(lib.bpm_step_generations(h, C.byref(st), 0, 3, None))
        _lib.check(lib.bpm_destroy(h))

    cycle()                                                    # the module loads lazily: warm up first
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(5):
        cycle()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free1 = torch.cuda.mem_get_info()[0]
    assert free1 >= free0 - 2 * (1 << 20), "5 cycles kept %d bytes" % (free0 - free1)
