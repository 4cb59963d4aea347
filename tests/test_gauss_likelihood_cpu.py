"""Gaussian likelihoods with a dense data covariance (targets.CudaGaussLikelihood), the parts that need no GPU:
bad input is refused on the host before any device is touched, the C-ABI refuses null and bad arguments, the
numpy reference the GPU tests use is scipy's multivariate_normal, and NVRTC compiles the model together with the
library's kernels for sm_100a at every shape test_gauss_likelihood_gpu.py runs.  The sources, cases and the
reference are shared with that file."""
import ctypes as C

import numpy as np
import pytest

# m(theta)_i = sum_q theta[q % d] * row[q % k] over q < max(d, k): every parameter and every column is read, with
# + and * only, so the numpy restatement below rounds exactly as the device does at fmad=False
ALLCOL_MEAN = r'''
__device__ double model_mean(const double* theta, const double* row) {
  const int nq = BPM_DIM > BPM_ROWLEN ? BPM_DIM : BPM_ROWLEN;
  double m = 0.0;
  for (int q = 0; q < nq; ++q) m = m + theta[q % BPM_DIM] * row[q % BPM_ROWLEN];
  return m;
}
'''

# NaN where theta[0] < 0, which the prior excludes; the prior is + - * / only
HALF_PLANE_MEAN = r'''
__device__ double model_mean(const double* theta, const double* row) {
  return sqrt(theta[0]) * row[0] + theta[1];
}
'''
HALF_PLANE_PRIOR = r'''
__device__ double ln_prior(const double* theta) {
  if (theta[0] < 0.0) return -INFINITY;
  return -0.5 * ((theta[1] - 0.25) * (theta[1] - 0.25)) / 3.0 + theta[0] * 0.125;
}
'''

# linear model m(theta) = A theta, with A = x[:, :d]
LINEAR_MEAN = r'''
__device__ double model_mean(const double* theta, const double* row) {
  double m = 0.0;
  for (int q = 0; q < BPM_DIM; ++q) m = m + theta[q] * row[q];
  return m;
}
'''

# Part A of the GPU file: (M, d, k).  M crosses the 16-row padding (16 | 17, 112 | 113) and the 128-column blocks
# (1000, 4096); d = 32 | 33 is the register / pointer SumTheta boundary, k = 9 rows are not staged.
A_CASES = [(1, 1, 1), (3, 4, 3), (16, 5, 9), (17, 33, 1), (112, 1, 3), (113, 4, 9), (1000, 5, 3), (1000, 33, 9),
           (4096, 4, 1), (4096, 33, 3)]
# Part D: (d, M) of the oracle steps
D_CASES = [(2, 50), (2, 1024), (5, 50), (5, 1024)]


def allcol_mean_np(theta, x):
    """ALLCOL_MEAN in numpy for rows theta[n, d] and x[M, k], the same operations in the same order."""
    theta = np.atleast_2d(theta)
    d, k = theta.shape[1], x.shape[1]
    m = np.zeros((theta.shape[0], x.shape[0]))
    for q in range(max(d, k)):
        m = m + theta[:, q % d][:, None] * x[:, q % k][None, :]
    return m


def half_plane_prior_np(theta):
    theta = np.atleast_2d(theta)
    t0, t1 = theta[:, 0], theta[:, 1]
    with np.errstate(invalid="ignore"):
        v = -0.5 * ((t1 - 0.25) * (t1 - 0.25)) / 3.0 + t0 * 0.125
    return np.where(t0 < 0.0, -np.inf, v)


def gauss_lnl_np(mean, y, B, c0):
    """ln L of predictions mean[n, M]: -0.5 (c0 + |(mean - y) B|^2), and the quadratic form's terms (for bounds)."""
    r = np.atleast_2d(mean) - y[None, :]
    z = r @ B
    return -0.5 * (c0 + np.sum(z * z, axis=1))


def exp_cov(t, ell, sigma=1.0, nugget=0.0):
    """Exponential-kernel covariance sigma^2 exp(-|t_i - t_j| / ell) + nugget I."""
    return sigma ** 2 * np.exp(-np.abs(t[:, None] - t[None, :]) / ell) + nugget * np.eye(t.size)


def random_cov(M, seed):
    """A well-conditioned dense covariance of mixed scales."""
    rs = np.random.RandomState(seed)
    t = np.sort(rs.uniform(0.0, 10.0, M))
    s = 10.0 ** rs.uniform(-1, 1, M)
    return exp_cov(t, 0.7, nugget=0.05) * s[:, None] * s[None, :]


def case_data(M, d, k, seed=0):
    """x [M, k], a centre theta0, and y = m(theta0) + correlated noise, with its covariance."""
    rs = np.random.RandomState(seed + 17 * M + d)
    x = rs.uniform(-1.0, 1.0, (M, k))
    theta0 = rs.uniform(-1.0, 1.0, d)
    cov = random_cov(M, seed + M)
    L = np.linalg.cholesky(cov)
    y = allcol_mean_np(theta0, x)[0] + L @ rs.randn(M)
    return x, y, cov, theta0


def _lik(**kw):
    from bipymc_b200 import targets
    M = 5
    x, y, cov, _ = case_data(M, 2, 1)
    args = dict(source=ALLCOL_MEAN, dim=2, x=x, y=y, cov=cov)
    args.update(kw)
    return targets.CudaGaussLikelihood(**args)


def _sym(a):
    return (a + a.T) / 2


@pytest.mark.parametrize("kw", [
    dict(source=ALLCOL_MEAN.encode()), dict(source=None), dict(dim=0), dict(dim=2.5), dict(dim=True),
    dict(x=np.zeros((5, 2, 1))), dict(x=np.zeros((0, 1))), dict(x=np.zeros((5, 0))), dict(x=[[0.0], [np.nan]] * 3),
    dict(x=np.full(5, np.inf)), dict(y=np.zeros(4)), dict(y=np.zeros((5, 1))), dict(y=[0, 0, 0, np.nan, 0]),
    dict(cov=np.eye(4)), dict(cov=np.eye(5)[:, :4]), dict(cov=np.where(np.eye(5) > 0, np.inf, 0.0)),
    dict(cov=np.eye(5) + 1e-9 * np.triu(np.ones((5, 5)), 1)),            # asymmetric
    dict(cov=-np.eye(5)), dict(cov=np.diag([1.0, 1.0, 1.0, 1.0, -1e-3])),   # not positive definite
    dict(cov=np.ones((5, 5))), dict(cov=np.diag([1.0, 1.0, 1.0, 1.0, 0.0])),  # singular
    dict(cov=np.diag([1.0, 1.0, 1.0, 1.0, 1e-13])),                          # singular by scipy's threshold
])
def test_bad_arguments_raise_value_error(kw):
    with pytest.raises(ValueError):
        _lik(**kw)


def test_singular_covariances_are_refused_as_scipy_refuses_them():
    from scipy.stats import multivariate_normal
    for cov in (np.ones((5, 5)), np.diag([1.0, 1.0, 1.0, 1.0, 1e-13]), _sym(np.outer(np.arange(5.0), np.arange(5.0)))):
        with pytest.raises(np.linalg.LinAlgError):
            multivariate_normal(np.zeros(5), cov)
        with pytest.raises(ValueError, match="positive definite"):
            _lik(cov=cov)
    multivariate_normal(np.zeros(5), np.diag([1.0, 1.0, 1.0, 1.0, 1e-8]))
    _lik(cov=np.diag([1.0, 1.0, 1.0, 1.0, 1e-8]))           # accepted by both


def test_too_many_rows_is_refused_before_the_covariance_is_read():
    from bipymc_b200 import targets
    with pytest.raises(ValueError, match="32768"):
        targets.CudaGaussLikelihood(ALLCOL_MEAN, 2, np.zeros(32769), np.zeros(32769), None)


def test_the_lower_triangle_is_used():
    lik = _lik()
    messy = lik.cov + 1e-14 * np.triu(np.ones_like(lik.cov), 1) * np.max(np.abs(lik.cov))
    other = _lik(cov=messy)
    assert np.array_equal(other.B, lik.B) and other.c0 == lik.c0
    assert np.all(np.tril(lik.B, -1) == 0.0)


def test_one_dimensional_x_is_one_value_per_row():
    lik = _lik(x=np.arange(5.0))
    assert lik.x.shape == (5, 1)


def test_more_than_one_rank_is_refused_before_the_device(monkeypatch):
    from bipymc_b200 import DeMc, DeMcMpi, DreamMpi, demc, samplers

    class _TwoRanks(demc._SingleComm):
        rank, size = 0, 2

    monkeypatch.setattr(demc, "_resolve_comm", lambda c: _TwoRanks())
    monkeypatch.setattr(samplers, "_resolve_comm", lambda c: _TwoRanks())
    monkeypatch.setattr(DeMcMpi, "_setup_device", lambda self: pytest.fail("the device was touched"))
    for cls in (DeMcMpi, DreamMpi):
        with pytest.raises(ValueError, match="one rank"):
            cls(lambda t: 0.0, np.zeros(2), n_chains=8, ln_like_cuda=_lik())
    with pytest.raises(ValueError, match="one rank"):
        DeMc(lambda t: 0.0, n_chains=8, ln_like_cuda=_lik())


@pytest.mark.parametrize("M", [1, 2, 17, 300, 1000])
def test_reference_is_scipy_multivariate_normal(M):
    from scipy.stats import multivariate_normal
    from bipymc_b200 import targets
    x, y, cov, theta0 = case_data(M, 3, 2)
    B, c0 = targets.CudaGaussLikelihood.factor(cov)
    rs = np.random.RandomState(M)
    for theta in theta0 + 0.3 * rs.randn(4, 3):
        mean = allcol_mean_np(theta, x)[0]
        want = multivariate_normal(mean, cov).logpdf(y)
        got = gauss_lnl_np(mean, y, B, c0)[0]
        assert abs(got - want) <= 1e-12 * max(1.0, abs(want)), (got, want)


def test_allcol_restatement_is_the_scalar_loop():
    rs = np.random.RandomState(1)
    for d, k in [(1, 1), (4, 9), (33, 3), (5, 9)]:
        theta, x = rs.randn(d), rs.randn(7, k)
        got = allcol_mean_np(theta, x)[0]
        for i, row in enumerate(x):
            m = 0.0
            for q in range(max(d, k)):
                m = m + theta[q % d] * row[q % k]
            assert got[i] == m


@pytest.mark.parametrize("case", range(len(A_CASES)))
def test_value_cases_compile_for_sm100a(case):
    from bipymc_b200 import targets
    M, d, k = A_CASES[case]
    x = np.zeros((M, k))
    targets.CudaGaussLikelihood(ALLCOL_MEAN, d, x, np.zeros(M), np.eye(M), fmad=False).compile()


def test_other_gpu_sources_compile_for_sm100a():
    from bipymc_b200 import targets
    for prior in (False, True):
        targets.CudaGaussLikelihood(HALF_PLANE_MEAN + (HALF_PLANE_PRIOR if prior else ""), 2, np.ones(64), np.zeros(64),
                                    np.eye(64), prior=prior, fmad=False).compile()
    for d, M in D_CASES:
        targets.CudaGaussLikelihood(ALLCOL_MEAN, d, np.zeros((M, 3)), np.zeros(M), np.eye(M), fmad=False).compile()
    targets.CudaGaussLikelihood(LINEAR_MEAN, 3, np.zeros((512, 3)), np.zeros(512), np.eye(512)).compile()


def test_cache_keys_on_the_shape_not_on_y_or_cov():
    from bipymc_b200 import targets
    src = ALLCOL_MEAN + "// cache key %d\n" % np.random.randint(1 << 30)
    x, y, cov, _ = case_data(40, 3, 2)

    def fresh(**kw):
        args = dict(source=src, dim=3, x=x, y=y, cov=cov, prior=False, fmad=True)
        args.update(kw)
        return targets.CudaGaussLikelihood(**args).compile() is False

    assert fresh()
    assert not fresh()                                            # same key: from the cache
    assert not fresh(y=y + 1.0, cov=2.0 * cov)                    # new data of the same shape
    assert fresh(x=x[:39], y=y[:39], cov=cov[:39, :39])           # M
    assert fresh(x=np.ones((40, 1)))                              # k
    assert fresh(fmad=False)
    assert fresh(dim=4)


def _abi():
    from bipymc_b200 import _lib
    return _lib.load()


def test_c_abi_refuses_null_and_bad_arguments():
    lib = _abi()
    M = 4
    x, y, B = np.zeros(M), np.zeros(M), np.eye(M)
    cached = C.c_int32(7)
    log = C.create_string_buffer(64)
    src = ALLCOL_MEAN.encode()
    p = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))          # noqa: E731
    assert lib.bpm_set_jit_gauss_target(None, src, p(x), M, 1, p(y), p(B), 1.0, 0, C.byref(cached), log, 64) != 0
    assert b"null handle" in lib.bpm_last_error() and cached.value == 0
    for args, why in [((None, 2, M, 1), b"null source"), ((src, 0, M, 1), b"dim"), ((src, 2, 0, 1), b"n_rows"),
                      ((src, 2, 32769, 1), b"n_rows"), ((src, 2, M, 0), b"row_len"),
                      ((b"__device__ double f(const double* t, const double* r) { return 0.0; }", 2, M, 1),
                       b"model_mean")]:
        assert lib.bpm_jit_compile_gauss(*args, 0, C.byref(cached), log, 64) != 0, args
        assert why in lib.bpm_last_error(), (args, lib.bpm_last_error())
    assert lib.bpm_jit_compile_gauss(src, 2, M, 1, 0, C.byref(cached), log, 64) == 0


def test_the_target_id_is_the_headers():
    import os
    from bipymc_b200 import _lib
    h = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "bipymc_b200.h")
    with open(h) as f:
        assert "#define BPM_TARGET_JIT_GAUSS %d " % _lib.TARGET_JIT_GAUSS in f.read()
