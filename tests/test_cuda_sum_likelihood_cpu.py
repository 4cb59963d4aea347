"""Per-observation CUDA likelihoods (targets.CudaSumLikelihood), the parts that need no GPU: NVRTC
compiles the user's terms together with the library's sum kernels for sm_100a, bad input is refused
on the host, and the numpy restatement of the summation order (used by the GPU tests to check the
device bit for bit) is sound.  The sources are shared with test_cuda_sum_likelihood_gpu.py."""
import math

import numpy as np
import pytest

CHUNK = 256      # rows per chunk (csrc/kernels_sum.cuh: kSumChunk)

# examples/ex_para_fit.py:39-55 per observation; row = (x, y, yerr)
LINEFIT_TERM = r'''
__device__ double ln_like_term(const double* theta, const double* row) {
  const double m = theta[0], b = theta[1], lnf = theta[2];
  const double model = m * row[0] + b;
  const double inv = 1.0 / (row[2] * row[2] + model * model * exp(2.0 * lnf));
  const double r = row[1] - model;
  return -0.5 * (r * r * inv - log(inv));
}
'''
LINEFIT_PRIOR = r'''
__device__ double ln_prior(const double* theta) {
  const double m = theta[0], b = theta[1], lnf = theta[2];
  return (-5.0 < m && m < 0.5 && 0.0 < b && b < 10.0 && -10.0 < lnf && lnf < 1.0) ? 0.0 : -INFINITY;
}
'''

# examples/ex_exp_fit.py:73-121 per observation; row = (t, y); theta = (tau, c_inf, c_0, leak, sigma)
EXPFIT_TERM = r'''
__device__ double ln_like_term(const double* th, const double* row) {
  const double m = th[1] + th[2] * -1.0 * exp(-row[0] / th[0]) - th[3] * row[0];
  const double r = m - row[1];
  return -0.5 * (r * r / th[4] - log(1.0 / th[4]));
}
'''
EXPFIT_PRIOR = r'''
__device__ double ln_prior(const double* th) {
  const double tau = th[0], c_inf = th[1], c_0 = th[2], leak = th[3], sigma = th[4];
  return (-5.0 < c_inf && c_inf < 5.0 && 1.0 < tau && tau < 50.0 && -1.0 < c_0 && c_0 < 1.0 &&
          -5.0 < leak && leak < 5.0 && 0.0 < sigma && sigma < 1.0) ? 0.0 : -INFINITY;
}
'''

# Gaussian polynomial fit with known errors, + - * / only: y = sum_q theta[q] x^q; row = (x, y, sigma)
POLY_TERM = r'''
__device__ double ln_like_term(const double* theta, const double* row) {
  double model = theta[BPM_DIM - 1];
  for (int q = BPM_DIM - 2; q >= 0; --q) model = model * row[0] + theta[q];
  const double r = (row[1] - model) / row[2];
  return -0.5 * (r * r);
}
'''


def poly_terms_np(theta, data):
    """POLY_TERM in numpy, the same operations in the same order (every one rounded: fmad=False)."""
    x, y, s = data[:, 0], data[:, 1], data[:, 2]
    model = np.full_like(x, theta[-1])
    for q in range(len(theta) - 2, -1, -1):
        model = model * x + theta[q]
    r = (y - model) / s
    return -0.5 * (r * r)


def sum_order(terms):
    """The library's summation order (csrc/kernels_sum.cuh): chunks of 256 rows padded with 0.0, a
    halving pairwise tree inside each chunk, then an adjacent-pair tree over the chunk partials padded
    with 0.0 to a power of two."""
    terms = np.asarray(terms, dtype=np.float64)
    M = terms.size
    nc = -(-M // CHUNK)
    a = np.zeros((nc, CHUNK))
    a.flat[:M] = terms
    while a.shape[1] > 1:
        h = a.shape[1] // 2
        a = a[:, :h] + a[:, h:]
    p = np.zeros(1 << (nc - 1).bit_length())
    p[:nc] = a[:, 0]
    while p.size > 1:
        p = p[0::2] + p[1::2]
    return p[0]


def poly_data(M, d, seed=7):
    rs = np.random.RandomState(seed)
    x = np.sort(rs.uniform(-1.0, 1.0, M))
    s = 0.05 + 0.1 * rs.rand(M)
    coef = np.arange(1, d + 1) * 0.3
    y = np.polyval(coef[::-1], x) + s * rs.randn(M)
    return np.stack([x, y, s], axis=1)


def linefit_rows():
    from bipymc_b200 import targets
    f = targets.LineFit()
    return np.stack([f.x, f.y, f.yerr], axis=1)


def expfit_rows(n=60):
    from bipymc_b200 import targets
    return np.stack(targets.expfit_data(n=n), axis=1)


@pytest.mark.parametrize("name", ["linefit", "linefit_prior", "expfit", "expfit_prior"])
def test_term_sources_compile_for_sm100a(name):
    from bipymc_b200 import targets
    src, dim, data = {"linefit": (LINEFIT_TERM, 3, linefit_rows()), "expfit": (EXPFIT_TERM, 5, expfit_rows())}[
        name.split("_")[0]]
    prior = name.endswith("_prior")
    if prior:
        src += LINEFIT_PRIOR if dim == 3 else EXPFIT_PRIOR
    lik = targets.CudaSumLikelihood(src, dim, data, prior=prior, fmad=False)
    lik.compile()
    assert lik.compile() is True          # the second compile of the same source comes from the process cache


def test_compile_error_names_the_user_line():
    from bipymc_b200 import targets
    src = ("__device__ double ln_like_term(const double* theta, const double* row) {\n"
           "  double a = theta[0];\n"
           "  return a * row[0] + ;\n"
           "}\n")
    with pytest.raises(targets.CudaCompileError) as e:
        targets.CudaSumLikelihood(src, 2, np.ones(10)).compile()
    assert "ln_like.cu(3)" in e.value.log


def test_prior_without_a_definition_is_a_compile_error():
    from bipymc_b200 import targets
    with pytest.raises(targets.CudaCompileError, match="ln_prior"):
        targets.CudaSumLikelihood(LINEFIT_TERM, 3, linefit_rows(), prior=True).compile()


def test_source_without_a_term_is_refused():
    from bipymc_b200 import _lib, targets
    with pytest.raises(_lib.BpmError, match="ln_like_term"):
        targets.CudaSumLikelihood("__device__ double ln_like(const double* t, const double* d) { return 0.0; }",
                                  2, np.ones(4)).compile()


@pytest.mark.parametrize("kw", [dict(source=LINEFIT_TERM.encode()), dict(source=None),
                                dict(dim=0), dict(dim=-3), dict(dim=2.5), dict(dim=True),
                                dict(data=[[0.0, np.nan]]), dict(data=[np.inf]), dict(data=np.zeros((2, 3, 1))),
                                dict(data=np.zeros(0)), dict(data=np.zeros((4, 0))), dict(data=np.float64(1.0)),
                                dict(data=["a", "b"])])
def test_bad_arguments_raise_value_error(kw):
    from bipymc_b200 import targets
    args = dict(source=LINEFIT_TERM, dim=3, data=linefit_rows())
    args.update(kw)
    with pytest.raises(ValueError):
        targets.CudaSumLikelihood(**args)


def test_one_dimensional_data_is_one_value_per_row():
    from bipymc_b200 import targets
    lik = targets.CudaSumLikelihood(LINEFIT_TERM, 3, np.arange(5.0))
    assert lik.data.shape == (5, 1)


def test_cache_keys_on_rows_row_length_fmad_and_prior():
    from bipymc_b200 import targets
    src = LINEFIT_TERM + LINEFIT_PRIOR + "// cache key %d\n" % np.random.randint(1 << 30)
    rows = np.ones((100, 3))

    def fresh(**kw):
        args = dict(source=src, dim=3, data=rows, prior=False, fmad=True)
        args.update(kw)
        return targets.CudaSumLikelihood(**args).compile() is False

    assert fresh()
    assert not fresh()                                        # same key: from the cache
    assert fresh(data=np.ones((101, 3)))                      # M
    assert fresh(data=np.ones((100, 4)))                      # k
    assert fresh(fmad=False)
    assert fresh(prior=True)
    assert not fresh(data=np.zeros((100, 3)))                 # the values are not part of the key


@pytest.mark.parametrize("M", [1, 31, CHUNK - 1, CHUNK, CHUNK + 1, 5 * CHUNK + 3, 100003])
def test_sum_order_agrees_with_fsum(M):
    rs = np.random.RandomState(M)
    t = rs.randn(M) * 10.0 ** rs.uniform(-3, 3, M)
    exact = math.fsum(t)
    scale = np.sum(np.abs(t))
    assert abs(sum_order(t) - exact) <= 4 * np.finfo(float).eps * max(1, math.log2(M)) * scale


def test_sum_order_of_small_cases_by_hand():
    assert sum_order([1.5]) == 1.5
    t = np.arange(1.0, 2 * CHUNK + 2)        # three chunks: ((c0 + c1) + (c2 + 0))
    c = [sum_order(t[i:i + CHUNK]) for i in range(0, t.size, CHUNK)]
    assert sum_order(t) == (c[0] + c[1]) + (c[2] + 0.0)
