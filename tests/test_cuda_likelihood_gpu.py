"""Run-time compiled CUDA likelihoods (targets.CudaLikelihood) on the GPU.

  * a source that restates a built-in target's arithmetic (calling its bpm:: function) gives the
    built-in's chains bit for bit -- in the fused d <= 4 kernel and on the split path (d = 5);
  * the kernels that ran are the ones the engine plans (launch counts by kind);
  * sources in the reference's own form (fmad=False) replay the reference's recorded draws to its
    golden histories, in the fused and the split kernels;
  * data past the shared-memory threshold (read from global memory) gives the same chains;
  * -inf rejects, NaN raises, and a second sampler takes the cached cubin."""
import numpy as np
import pytest

from test_cuda_likelihood_cpu import (BANANA_SAME, EXPFIT_SAME, LINEFIT_PER_TERM, LINEFIT_SAME, banana_data,
                                      expfit_data, linefit_data)
from test_replay_parity_gpu import ALL_CASES, check_against_reference, launches_by_kind, oracle_traces

pytestmark = pytest.mark.gpu


def _never(theta, **kw):
    raise AssertionError("ln_like_fn must not be called when ln_like_cuda is given")


def _run(cls, fn, theta0, N, G, fused=1, seed=11, **kw):
    np.random.seed(5)
    s = cls(fn, np.asarray(theta0, dtype=float), n_chains=N, seed=seed, fused=fused, **kw)
    s.run_mcmc(N * (G + 1))
    return s


def _assert_same_chains(a, b):
    import torch
    d = a.dim
    ha, hb = a._hist.tensor()[:, :, :d], b._hist.tensor()[:, :, :d]
    assert ha.shape == hb.shape
    bad = [t for t in range(ha.shape[0]) if not torch.equal(ha[t], hb[t])]
    assert not bad, "generations with differing chains: %r" % bad[:5]
    assert torch.equal(a._lnl, b._lnl)
    assert (a.n_accepted, a.n_rejected) == (b.n_accepted, b.n_rejected)
    if hasattr(a, "p_cr"):
        assert np.array_equal(a.p_cr, b.p_cr)


def _builtin_case(name):
    from bipymc_b200 import DeMcMpi, DreamMpi, targets
    dream = dict(n_cr_gen=3, burnin_gen=1000)
    if name == "banana_dream":
        return DreamMpi, targets.Banana_2D(sigma1=1.0, sigma2=1.0).ln_like, BANANA_SAME, banana_data(), \
            [0.0, 0.0], dict(varepsilon=1.0, **dream)
    if name == "banana_demc":
        return DeMcMpi, targets.Banana_2D(sigma1=1.0, sigma2=1.0).ln_like, BANANA_SAME, banana_data(), \
            [0.0, 0.0], dict(varepsilon=1.0)
    if name == "linefit_dream":
        return DreamMpi, targets.LineFit().ln_like, LINEFIT_SAME, linefit_data(), [-0.8, 4.5, 0.2], \
            dict(varepsilon=1e-2, **dream)
    if name == "expfit_dream_d5":
        return DreamMpi, targets.ExpFit().ln_like, EXPFIT_SAME, expfit_data(), [12.0, 1.5, 0.6, 1e-3, 2e-3], \
            dict(varepsilon=np.asarray([1e-2, 1e-2, 1e-3, 1e-8, 1e-9]) * 1e-2, **dream)     # ex_exp_fit.py:135
    raise KeyError(name)


@pytest.mark.parametrize("name", ["banana_dream", "banana_demc", "linefit_dream", "expfit_dream_d5"])
def test_same_arithmetic_as_builtin_gives_same_chains(name, monkeypatch):
    from bipymc_b200 import DeMcMpi, targets
    cls, builtin, src, data, theta0, kw = _builtin_case(name)
    N, G = 2000, 25
    ref = _run(cls, builtin, theta0, N, G, **kw)
    assert ref._mode() == "device"

    def no_split(*a, **k):
        raise AssertionError("the CUDA likelihood left the library (_split_generation)")
    monkeypatch.setattr(DeMcMpi, "_split_generation", no_split)
    from bipymc_b200 import _lib
    lik = targets.CudaLikelihood(src, len(theta0), data, fmad=True)
    np.random.seed(5)
    s = cls(_never, np.asarray(theta0, dtype=float), n_chains=N, seed=11, fused=1, ln_like_cuda=lik, **kw)
    assert s._mode() == "device"
    _lib.check(s._libh.bpm_profile(s._handle, 1))
    s.run_mcmc(N * (G + 1))
    k = launches_by_kind(s)
    if len(theta0) <= 4:
        assert k["fused_phase"] == 2 * G and k["propose"] == 0 and k["likelihood"] == 0, k
    else:
        assert k["propose"] == k["likelihood"] == k["accept"] == 2 * G and k["fused_phase"] == 0, k
    _assert_same_chains(ref, s)


@pytest.mark.parametrize("algo", ["dream", "demc"])
def test_fused_and_split_agree(algo):
    from bipymc_b200 import DeMcMpi, DreamMpi, targets
    cls = DreamMpi if algo == "dream" else DeMcMpi
    kw = dict(n_cr_gen=3, burnin_gen=1000) if algo == "dream" else {}
    lik = targets.CudaLikelihood(LINEFIT_PER_TERM, 3, linefit_data(), fmad=True)
    runs = [_run(cls, _never, [-0.8, 4.5, 0.2], 1500, 20, fused=f, varepsilon=1e-2, ln_like_cuda=lik, **kw)
            for f in (1, 0)]
    _assert_same_chains(*runs)


# The reference's own forms (fmad=False: every + - * / rounded like numpy)
BANANA_REF = r'''
__device__ double ln_like(const double* y, const double* p) {
  // p = log_of_pdf, a, b, mu0, mu1, U00, U01, U10, U11, c0   (banana_rv.py:26-37, scipy's logpdf)
  const double a = p[1], b = p[2];
  const double x1 = y[0] / a;
  const double x2 = (y[1] - b * (x1 * x1 + a * a)) * a;
  const double d0 = x1 - p[3], d1 = x2 - p[4];
  const double w0 = d0 * p[5] + d1 * p[7], w1 = d0 * p[6] + d1 * p[8];
  const double lp = -0.5 * (p[9] + (w0 * w0 + w1 * w1));
  return log(exp(lp));
}
'''

GAUSS_REF = r'''
__device__ double ln_like(const double* x, const double* p) {
  // p = c0, mu[d], U[d][d] row-major   (d100_gauss.py:29-35: np.log(multivariate_normal.pdf))
  const int d = BPM_DIM;
  const double* mu = p + 1;
  const double* U = p + 1 + d;
  double maha = 0.0;
  for (int j = 0; j < d; ++j) {
    double w = 0.0;
    for (int i = 0; i < d; ++i) w += (x[i] - mu[i]) * U[i * d + j];
    maha += w * w;
  }
  return log(exp(-0.5 * (p[0] + maha)));
}
'''


def _reference_form(target):
    from bipymc_b200 import targets
    if target == "banana":
        return BANANA_REF, banana_data()
    if target == "linefit":
        return LINEFIT_PER_TERM, linefit_data()
    if target.startswith("gauss"):
        g = targets.Gauss_100D(dim=int(target[5:]))
        assert g.rv_100d.U.shape == (g.dim, g.dim)
        return GAUSS_REF, np.concatenate([[g.rv_100d.c0], g.rv_100d.mean, g.rv_100d.U.ravel()])
    raise KeyError(target)


@pytest.mark.parametrize("fused", [1, 0], ids=["fused", "split"])
@pytest.mark.parametrize("name", ["linefit_dream", "banana_demc", "banana_dream_odd", "gauss7_dream_noshuffle"])
def test_replay_parity_reference_form(name, fused):
    from bipymc_b200 import DeMcMpi, DreamMpi, _lib, targets
    case = ALL_CASES[name]
    osampler, traces = oracle_traces(name)
    src, data = _reference_form(case["target"])
    theta0 = np.asarray(case["theta_0"], dtype=float)
    lik = targets.CudaLikelihood(src, len(theta0), data, fmad=False)
    cls = DreamMpi if case["algo"] == "dream" else DeMcMpi
    np.random.seed(case["seed"])
    s = cls(_never, theta0, n_chains=case["n_chains"], fused=fused, ln_like_cuda=lik, **case["ctor_kwargs"])
    _lib.check(s._libh.bpm_profile(s._handle, 1))
    sink = []
    s.run_mcmc(case["n"], _replay=traces, _trace=sink, **case["run_kwargs"])
    k = launches_by_kind(s)
    gens = len(traces)
    if fused and len(theta0) <= 4:
        assert k["fused_phase"] == 2 * gens and k["propose"] == 0, k
    else:
        assert k["fused_phase"] == 0 and k["propose"] == k["likelihood"] == k["accept"] == 2 * gens, k
    check_against_reference(name, s, sink, traces, osampler)


# data[0] = M, then x[M], y[M], yerr[M]; whatever follows is padding the source never reads
LINEFIT_HEADER = r'''
__device__ double ln_like(const double* theta, const double* data) {
  const int M = (int)data[0];
  return bpm::linefit_lnl(data + 1, data + 1 + M, data + 1 + 2 * M, M, theta[0], theta[1], theta[2]);
}
'''


@pytest.mark.parametrize("fused", [1, 0], ids=["fused", "split"])
def test_data_past_the_shared_memory_threshold(fused):
    from bipymc_b200 import DreamMpi, targets
    base = np.concatenate([[50.0], linefit_data()])
    padded = np.concatenate([base, np.zeros(5000)])          # > 4096 doubles: read from global memory
    runs = [_run(DreamMpi, _never, [-0.8, 4.5, 0.2], 1500, 20, fused=fused, varepsilon=1e-2, n_cr_gen=3,
                 burnin_gen=1000, ln_like_cuda=targets.CudaLikelihood(LINEFIT_HEADER, 3, d)) for d in (base, padded)]
    _assert_same_chains(*runs)


HALF_PLANE = r'''
__device__ double ln_like(const double* t, const double* data) {
  if (t[0] < 0.0) return -INFINITY;          // prior: theta_0 >= 0
  return -0.5 * ((t[0] - 0.2) * (t[0] - 0.2) + t[1] * t[1]);
}
'''


@pytest.mark.parametrize("fused", [1, 0], ids=["fused", "split"])
def test_minus_inf_outside_the_prior_is_rejected(fused):
    from bipymc_b200 import DreamMpi, targets
    s = _run(DreamMpi, _never, [0.5, 0.0], 1000, 30, fused=fused, varepsilon=1e-2, n_cr_gen=3, burnin_gen=1000,
             ln_like_cuda=targets.CudaLikelihood(HALF_PLANE, 2))
    h = s._hist.tensor()[:, :, :2].cpu().numpy()
    assert (h[:, :, 0] >= 0.0).all()
    assert np.isfinite(s._lnl.cpu().numpy()).all()
    assert 0 < s.n_accepted < s.n_accepted + s.n_rejected


def test_nan_raises():
    from bipymc_b200 import DeMcMpi, targets
    src = "__device__ double ln_like(const double* t, const double* d) { return t[0] > 1e300 ? 0.0 : NAN; }\n"
    s = DeMcMpi(_never, np.zeros(2), n_chains=64, seed=1, ln_like_cuda=targets.CudaLikelihood(src, 2))
    with pytest.raises(ValueError, match="probabilities contain NaN"):
        s.run_mcmc(64 * 4)


def test_second_sampler_takes_the_cached_cubin():
    from bipymc_b200 import DeMcMpi, targets
    src = LINEFIT_SAME + "// cache probe %d\n" % np.random.randint(1 << 30)
    s1 = DeMcMpi(_never, [-0.8, 4.5, 0.2], n_chains=64, seed=1,
                 ln_like_cuda=targets.CudaLikelihood(src, 3, linefit_data()))
    s2 = DeMcMpi(_never, [-0.8, 4.5, 0.2], n_chains=64, seed=1,
                 ln_like_cuda=targets.CudaLikelihood(src, 3, linefit_data()))
    assert s1._jit_from_cache is False and s2._jit_from_cache is True


def test_dimension_mismatch_is_refused():
    from bipymc_b200 import DeMcMpi, targets
    with pytest.raises(ValueError, match="dimension"):
        DeMcMpi(_never, np.zeros(2), n_chains=64, ln_like_cuda=targets.CudaLikelihood(LINEFIT_SAME, 3))
