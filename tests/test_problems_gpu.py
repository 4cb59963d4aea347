"""Several problems in one sampler (targets.CudaLikelihoodSet) on the GPU.

  * the contract: problem g of a multi-problem run equals a single-problem sampler with n chains, data
    row g, key problem_seeds[g] and the same initial states, bit for bit (history, cached ln L, CR state,
    counters), for DREAM and DE-MC, odd and even n, fused and split at d = 3, and the split path at d = 5;
  * P = 1 equals an ordinary CudaLikelihood sampler with the same seed;
  * launches per generation do not depend on P;
  * no cross-talk: 1000 linear-Gaussian problems each match their own analytic posterior;
  * -inf and NaN in one problem, checkpoints, and the refused options."""
import ctypes as C

import numpy as np
import pytest

from test_cuda_likelihood_cpu import EXPFIT_SAME, LINEFIT_PER_TERM
from test_problems_cpu import LINE_GAUSS, expfit_set, linefit_set
from test_replay_parity_gpu import launches_by_kind

pytestmark = pytest.mark.gpu

P = 7
LINEFIT_THETA0 = [-0.9, 4.3, -0.7]
EXPFIT_THETA0 = [12.0, 1.5, 0.6, 1e-3, 2e-3]


def _never(theta, **kw):
    raise AssertionError("ln_like_fn must not be called when ln_like_cuda is given")


def _multi(cls, src, dim, data, theta0, n, seed=11, varepsilon=1e-4, **kw):
    from bipymc_b200 import targets
    np.random.seed(5)
    lik = targets.CudaLikelihoodSet(src, dim, data, fmad=False)
    return cls(_never, np.asarray(theta0, dtype=float), n_chains=n, seed=seed, ln_like_cuda=lik,
               varepsilon=varepsilon, **kw)


def _single_like(ms, cls, src, dim, g, **kw):
    """Problem g of multi-problem sampler ms as a sampler of its own, started from the same states."""
    from bipymc_b200 import targets
    n = ms.n_chains
    lik = targets.CudaLikelihood(src, dim, ms._ln_like_cuda.data[g], fmad=False)
    s = cls(_never, np.zeros(dim), n_chains=n, seed=ms.problem_seeds[g], ln_like_cuda=lik, **kw)
    x0 = ms._hist.tensor()[:1, g * n:(g + 1) * n, :dim].cpu().numpy()
    s.load_history(x0)
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


CASES = {"linefit_d3_fused": (LINEFIT_PER_TERM, 3, linefit_set, LINEFIT_THETA0, 1e-3, 1),
         "linefit_d3_split": (LINEFIT_PER_TERM, 3, linefit_set, LINEFIT_THETA0, 1e-3, 0),
         "expfit_d5": (EXPFIT_SAME, 5, expfit_set, EXPFIT_THETA0, 1e-8, 1)}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("n", [33, 64])
@pytest.mark.parametrize("algo", ["dream", "demc"])
def test_each_problem_equals_its_single_problem_sampler(case, n, algo):
    from bipymc_b200 import DeMcMpi, DreamMpi
    src, dim, data_fn, theta0, var, fused = CASES[case]
    cls = DreamMpi if algo == "dream" else DeMcMpi
    # CR adaptation switches on after 3 rows and off at generation 14; gamma jumps every 5 / 10 generations
    kw = dict(n_cr_gen=3, burnin_gen=14) if algo == "dream" else {}
    ms = _multi(cls, src, dim, data_fn(P), theta0, n, varepsilon=var, fused=fused, **kw)
    singles = [_single_like(ms, cls, src, dim, g, fused=fused, **kw) for g in range(P)]
    G = 26
    ms.run_mcmc(n * (G + 1))
    assert ms._hist.length == G + 1
    assert np.all(ms.n_accepted > 0)
    for g, s in enumerate(singles):
        s.run_mcmc(n * (G + 1))
        _assert_problem_equal(ms, g, s, algo == "dream")
    # the problems differ from each other: their data do
    h = ms._hist.tensor()[-1, :, :dim].cpu().numpy()
    assert not np.array_equal(h[:n], h[n:2 * n])


@pytest.mark.parametrize("algo", ["dream", "demc"])
def test_one_problem_equals_an_ordinary_sampler(algo):
    from bipymc_b200 import DeMcMpi, DreamMpi, targets
    cls = DreamMpi if algo == "dream" else DeMcMpi
    kw = dict(n_cr_gen=3, burnin_gen=14) if algo == "dream" else {}
    data = linefit_set(1)
    ms = _multi(cls, LINEFIT_PER_TERM, 3, data, LINEFIT_THETA0, 40, varepsilon=1e-3, **kw)
    np.random.seed(5)
    s = cls(_never, np.asarray(LINEFIT_THETA0), n_chains=40, seed=11, varepsilon=1e-3,
            ln_like_cuda=targets.CudaLikelihood(LINEFIT_PER_TERM, 3, data[0], fmad=False), **kw)
    assert ms.problem_seeds == [11]
    ms.run_mcmc(40 * 21)
    s.run_mcmc(40 * 21)
    _assert_problem_equal(ms, 0, s, algo == "dream")


@pytest.mark.parametrize("case", ["linefit_d3_fused", "expfit_d5"])
def test_launches_per_generation_do_not_depend_on_p(case):
    from bipymc_b200 import DreamMpi, _lib
    src, dim, data_fn, theta0, var, _ = CASES[case]
    G = 8
    counts = []
    for n_prob in (P, 1000):
        ms = _multi(DreamMpi, src, dim, data_fn(n_prob), theta0, 32, varepsilon=var, n_cr_gen=3, burnin_gen=100)
        _lib.check(ms._libh.bpm_profile(ms._handle, 1))
        ms.run_mcmc(32 * (G + 1))
        counts.append(launches_by_kind(ms))
    assert counts[0] == counts[1], counts
    k = counts[0]
    assert k["split"] == G and k["cr_reduce"] == G, k
    if dim <= 4:
        assert k["fused_phase"] == 2 * G and k["propose"] == k["likelihood"] == k["accept"] == 0, k
    else:
        assert k["fused_phase"] == 0 and k["propose"] == k["likelihood"] == k["accept"] == 2 * G, k


def test_no_cross_talk_at_scale():
    """1000 problems x 64 chains, y = a_g + b_g x + N(0, sigma^2) with known sigma: every problem's
    posterior is Gaussian with its own mean and covariance (flat prior inside a wide box)."""
    from bipymc_b200 import DreamMpi
    n_prob, n, M = 1000, 64, 20
    rs = np.random.RandomState(7)
    x = np.linspace(-1.0, 1.0, M)
    a, b = rs.uniform(-5, 5, n_prob), rs.uniform(-3, 3, n_prob)
    sig = 0.3 + 0.2 * rs.rand(n_prob, M)
    y = a[:, None] + b[:, None] * x[None] + sig * rs.randn(n_prob, M)
    data = np.concatenate([np.tile(x, (n_prob, 1)), y, sig], axis=1)
    X = np.stack([np.ones(M), x], axis=1)
    mean, sd = np.zeros((n_prob, 2)), np.zeros((n_prob, 2))
    for g in range(n_prob):
        W = 1.0 / sig[g] ** 2
        cov = np.linalg.inv(X.T @ (W[:, None] * X))
        mean[g] = cov @ (X.T @ (W * y[g]))
        sd[g] = np.sqrt(np.diag(cov))
    ms = _multi(DreamMpi, LINE_GAUSS, 2, data, mean, n, varepsilon=0.01, n_cr_gen=5, burnin_gen=200)
    G = 400
    ms.run_mcmc(n * (G + 1))
    m, s, _ = ms.param_est(n * (G // 2))
    assert m.shape == s.shape == (n_prob, 2)
    z = np.abs(m - mean) / sd
    assert z.max() < 0.35, (z.max(), np.unravel_index(z.argmax(), z.shape))
    np.testing.assert_allclose(s, sd, rtol=0.2)
    md, sdd = ms.param_est_device(n * (G // 2))
    np.testing.assert_allclose(md, m, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(sdd, s, rtol=1e-9)
    assert ms.rhat().shape == (n_prob, 2) and np.all(ms.rhat() < 1.2)
    acc = ms.acceptance_fraction
    assert acc.shape == (n_prob,) and np.all((acc > 0.05) & (acc < 0.95))
    assert ms.super_chain.shape == (n_prob, n * (G + 1), 2)
    assert len(ms.am_chains) == n_prob * n


BOUNDED = r'''
__device__ double ln_like(const double* t, const double* data) {
  if (t[0] > data[0]) return -INFINITY;           // problem-specific prior bound
  if (data[1] != 0.0) return NAN;
  return -0.5 * (t[0] * t[0] + t[1] * t[1]);
}
'''


def test_minus_inf_stays_in_its_problem():
    from bipymc_b200 import DreamMpi
    data = np.array([[100.0, 0.0]] * P)
    data[3, 0] = 0.0
    ms = _multi(DreamMpi, BOUNDED, 2, data, [-0.5, 0.0], 32, varepsilon=1e-2)
    ms.run_mcmc(32 * 61)
    h = ms._hist.tensor()[:, :, :2].cpu().numpy().reshape(-1, P, 32, 2)
    assert (h[:, 3, :, 0] <= 0.0).all()
    assert all((h[:, g, :, 0] > 0.0).any() for g in range(P) if g != 3)
    assert np.isfinite(ms._lnl.cpu().numpy()).all()


def test_nan_in_one_problem_raises():
    from bipymc_b200 import DeMcMpi
    data = np.array([[100.0, 0.0]] * P)
    data[2, 1] = 1.0
    ms = _multi(DeMcMpi, BOUNDED, 2, data, [-0.5, 0.0], 32, varepsilon=1e-2)
    with pytest.raises(ValueError, match="probabilities contain NaN"):
        ms.run_mcmc(32 * 4)


@pytest.mark.parametrize("ext", [".h5", ".npz"])
def test_checkpoint_resumes_bit_for_bit(tmp_path, ext):
    from bipymc_b200 import DreamMpi
    path = str(tmp_path / ("ck" + ext))
    kw = dict(n_cr_gen=3, burnin_gen=30)
    a = _multi(DreamMpi, LINEFIT_PER_TERM, 3, linefit_set(P), LINEFIT_THETA0, 33, seed=[5, 9, 2, 7, 1, 3, 8],
               varepsilon=1e-3, **kw)
    a.run_mcmc(33 * 13)
    a.save_state(path)
    a.run_mcmc(33 * 13)
    b = _multi(DreamMpi, LINEFIT_PER_TERM, 3, linefit_set(P), LINEFIT_THETA0, 33, seed=0, varepsilon=1e-3, **kw)
    b.load_state(path)
    assert b.problem_seeds == [5, 9, 2, 7, 1, 3, 8]
    np.testing.assert_array_equal(b.p_cr.shape, (P, 3))
    b.run_mcmc(33 * 13)
    np.testing.assert_array_equal(a._hist.tensor()[:, :, :3].cpu().numpy(), b._hist.tensor()[:, :, :3].cpu().numpy())
    np.testing.assert_array_equal(a._lnl.cpu().numpy(), b._lnl.cpu().numpy())
    np.testing.assert_array_equal(a.p_cr, b.p_cr)
    np.testing.assert_array_equal(a.n_accepted, b.n_accepted)


def test_refused_options():
    from bipymc_b200 import DreamMpi, _lib
    ms = _multi(DreamMpi, LINEFIT_PER_TERM, 3, linefit_set(P), LINEFIT_THETA0, 32, varepsilon=1e-3)
    with pytest.raises(NotImplementedError):
        ms.track_covariance()
    with pytest.raises(NotImplementedError):
        ms.rhat_history()
    with pytest.raises(ValueError, match="_replay"):
        ms.run_mcmc(32 * 3, _replay=[{}])
    lib, h = ms._libh, ms._handle
    st = ms._state(None)
    s = ms._stream()
    buf = np.zeros(64)
    calls = {
        "bpm_set_target": lambda: lib.bpm_set_target(h, _lib.TARGET_LINEFIT, _lib.dptr(buf), 1),
        "bpm_set_jit_target": lambda: lib.bpm_set_jit_target(h, b"x", _lib.dptr(buf), 1, 1, None, None, 0),
        "bpm_set_cr_state": lambda: lib.bpm_set_cr_state(h, _lib.dptr(buf), None, None),
        "bpm_get_cr_state": lambda: lib.bpm_get_cr_state(h, _lib.dptr(buf), None, None),
        "bpm_begin_generation": lambda: lib.bpm_begin_generation(h, C.byref(st), 0, None, s),
        "bpm_step_generation_replay": lambda: lib.bpm_step_generation_replay(h, C.byref(st), C.byref(_lib.Replay()),
                                                                             0, None, s),
        "bpm_dump_draws": lambda: lib.bpm_dump_draws(h, C.byref(st), 0, C.byref(_lib.Replay()), None, s),
        "bpm_generations_host": lambda: lib.bpm_generations_host(h, buf.ctypes.data, buf.ctypes.data, 0, 0, 1),
        "bpm_generations_host_sharded": lambda: lib.bpm_generations_host_sharded(
            h, C.byref(st), buf.ctypes.data, buf.ctypes.data, 0, 1, s),
        "bpm_omega_track": lambda: lib.bpm_omega_track(h, 1),
        "bpm_cov_track": lambda: lib.bpm_cov_track(h, 1),
        "bpm_rhat": lambda: lib.bpm_rhat(h, C.byref(st), -1, buf.ctypes.data, s),
        "bpm_set_problems": lambda: lib.bpm_set_problems(h, 1, (C.c_uint64 * 1)(0)),
    }
    for name, call in calls.items():
        assert call() != 0, name
        assert b"multi-problem" in lib.bpm_last_error(), (name, lib.bpm_last_error())
    # the other likelihoods cannot be set on a multi-problem handle, and bpm_eval_lnl wants whole problems
    rows = ms._X[:P + 1]
    out = ms._lnl[:P + 1].clone()
    assert lib.bpm_eval_lnl(h, rows.data_ptr(), P + 1, out.data_ptr(), s) != 0
