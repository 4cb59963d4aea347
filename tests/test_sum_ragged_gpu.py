"""Per-observation likelihoods for datasets of different lengths in one sampler (targets.CudaSumLikelihoodSet given
a list of arrays) on the GPU.

  * the per-problem contract: problem g of a run equals a single-problem CudaSumLikelihood sampler with n chains,
    its own M_g rows, key problem_seeds[g] and the same initial states, bit for bit (history, cached ln L, CR
    state, counters), for DREAM and DE-MC, odd and even n, d = 3 and 5, with problems of one and of several groups
    of chunks in the same launch, one shorter than a group, and a prior that is -inf over part of one problem's
    posterior;
  * the order contract: bpm_eval_lnl of problem g's rows equals the numpy restatement of the summation order over
    problem g's terms bit for bit, whatever the batch per problem;
  * the ragged set and the rectangular set padded with masked rows give the same ln L;
  * launches per generation depend neither on P nor on the lengths;
  * NaN in one problem, and checkpoints."""
import numpy as np
import pytest

from test_cuda_sum_likelihood_cpu import CHUNK, POLY_TERM, poly_data, poly_terms_np, sum_order
from test_problems_gpu import _assert_problem_equal
from test_replay_parity_gpu import launches_by_kind

pytestmark = pytest.mark.gpu

# one group and several, a problem shorter than a group, chunk edges, and a few others
LENGTHS = [1, CHUNK - 1, CHUNK, CHUNK + 1, 4097, 100003] + np.random.RandomState(1).randint(2, 5000, 3).tolist()
# -inf for part of the box: problem BOUNDARY's posterior straddles theta[0] = 1
PRIOR = r'''
__device__ double ln_prior(const double* t) { return t[0] < 1.0 ? 0.0 : -INFINITY; }
'''
BOUNDARY = 4


def _never(theta, **kw):
    raise AssertionError("ln_like_fn must not be called when ln_like_cuda is given")


def _poly_ragged(lengths, d, shift=None):
    """POLY_TERM rows (x, y, sigma) of y = sum_q 0.3 (q + 1) x^q + noise, problem g of lengths[g] rows; shift[g]
    is added to y (to theta[0])."""
    out = [poly_data(m, d, seed=7 + g) for g, m in enumerate(lengths)]
    for g, v in (shift or {}).items():
        out[g][:, 1] += v
    return out


def _theta0(parts, d, shift=None):
    t = np.tile(np.arange(1, d + 1) * 0.3, (len(parts), 1))
    for g, v in (shift or {}).items():
        t[g, 0] += v
    return t


def _multi(cls, src, dim, data, theta0, n, prior=False, seed=11, varepsilon=1e-4, **kw):
    from bipymc_b200 import targets
    np.random.seed(5)
    lik = targets.CudaSumLikelihoodSet(src, dim, data, prior=prior, fmad=False)
    return cls(_never, np.asarray(theta0, dtype=float), n_chains=n, seed=seed, ln_like_cuda=lik,
               varepsilon=varepsilon, **kw)


def _problem_rows(lik, g):
    off = np.concatenate([[0], np.cumsum(lik.n_rows)])
    return lik.data[off[g]:off[g + 1]]


def _eval(s, theta):
    """bpm_eval_lnl of host rows theta[n, d] on sampler s (rows problem-major, n / P each)."""
    import torch
    rows = torch.zeros((theta.shape[0], s._ld), dtype=torch.float64, device=s._device)
    rows[:, :s.dim] = torch.from_numpy(np.ascontiguousarray(theta)).to(s._device)
    out = s._eval_lnl_rows(rows)
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("d", [3, 5])
@pytest.mark.parametrize("n", [33, 64])
@pytest.mark.parametrize("algo", ["dream", "demc"])
def test_each_problem_equals_its_single_problem_sampler(d, n, algo):
    from bipymc_b200 import DeMcMpi, DreamMpi, targets
    cls = DreamMpi if algo == "dream" else DeMcMpi
    kw = dict(n_cr_gen=3, burnin_gen=14) if algo == "dream" else {}
    shift = {BOUNDARY: 0.695}        # theta[0] = 0.995, posterior sd ~ 0.003 at M = 4097: by the prior's edge
    parts = _poly_ragged(LENGTHS, d, shift)
    # initial states theta_0 + N(0, varepsilon): sd 1e-3, all inside the prior
    ms = _multi(cls, POLY_TERM + PRIOR, d, parts, _theta0(parts, d, shift), n, prior=True, varepsilon=1e-6, **kw)
    lik = ms._ln_like_cuda
    assert lik.n_rows.tolist() == LENGTHS
    singles = []
    for g in range(len(LENGTHS)):
        one = targets.CudaSumLikelihood(lik.source, d, _problem_rows(lik, g), prior=True, fmad=False)
        s = cls(_never, np.zeros(d), n_chains=n, seed=ms.problem_seeds[g], ln_like_cuda=one, **kw)
        s.load_history(ms._hist.tensor()[:1, g * n:(g + 1) * n, :d].cpu().numpy())
        singles.append(s)
    G = 26
    ms.run_mcmc(n * (G + 1))
    assert ms._hist.length == G + 1
    for g, s in enumerate(singles):
        s.run_mcmc(n * (G + 1))
        _assert_problem_equal(ms, g, s, algo == "dream")
    # the prior's edge was proposed past in problem BOUNDARY: its rejections include -inf proposals
    h = ms._hist.tensor()[:, BOUNDARY * n:(BOUNDARY + 1) * n, 0].cpu().numpy()
    assert (h < 1.0).all() and h.max() > 0.99


def test_order_contract_bit_for_bit():
    from bipymc_b200 import DeMcMpi
    d = 3
    parts = _poly_ragged(LENGTHS, d)
    P = len(parts)
    ms = _multi(DeMcMpi, POLY_TERM, d, parts, _theta0(parts, d), 8)
    rs = np.random.RandomState(3)
    B = 4096                                                  # rows per problem of the largest batch
    th = np.arange(1, d + 1) * 0.3 + 0.01 * rs.randn(P, B, d)
    got = {b: np.concatenate([_eval(ms, th[:, i:i + b].reshape(-1, d)).reshape(P, -1)
                              for i in range(0, B, b)], axis=1) for b in (1, 7, B)}
    assert np.array_equal(got[1], got[B]) and np.array_equal(got[7], got[B])
    for g, m in enumerate(LENGTHS):
        pick = np.arange(0, B, 1 if m < 1000 else 256)
        ref = np.array([sum_order(poly_terms_np(th[g, i], parts[g])) for i in pick])
        assert np.array_equal(got[B][g, pick], ref), g


# POLY_TERM with a mask column: rows whose last value is 0.0 add nothing
MASKED = r'''
__device__ double ln_like_term(const double* theta, const double* row) {
  if (row[BPM_ROWLEN - 1] == 0.0) return 0.0;
  double model = theta[BPM_DIM - 1];
  for (int q = BPM_DIM - 2; q >= 0; --q) model = model * row[0] + theta[q];
  const double r = (row[1] - model) / row[2];
  return -0.5 * (r * r);
}
'''


def test_ragged_equals_padded_with_mask():
    from bipymc_b200 import DeMcMpi
    d = 3
    parts = [np.concatenate([p, np.ones((p.shape[0], 1))], axis=1) for p in _poly_ragged(LENGTHS, d)]
    P, M = len(parts), max(LENGTHS)
    padded = np.zeros((P, M, 4))
    for g, p in enumerate(parts):
        padded[g, :p.shape[0]] = p
    rag = _multi(DeMcMpi, MASKED, d, parts, _theta0(parts, d), 8)
    rect = _multi(DeMcMpi, MASKED, d, padded, _theta0(parts, d), 8)
    assert rag._ln_like_cuda.n_rows is not None and rect._ln_like_cuda.data.shape == (P, M, 4)
    th = np.arange(1, d + 1) * 0.3 + 0.01 * np.random.RandomState(4).randn(P * 64, d)
    a, b = _eval(rag, th), _eval(rect, th)
    assert np.isfinite(a).all()
    np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("d", [3, 5])
def test_launches_per_generation_do_not_depend_on_p_or_lengths(d):
    from bipymc_b200 import DreamMpi, _lib
    G = 8
    counts = []
    rs = np.random.RandomState(2)
    for lengths in (LENGTHS, np.exp(rs.uniform(np.log(100), np.log(20000), 1000)).astype(int).tolist()):
        parts = _poly_ragged(lengths, d)
        ms = _multi(DreamMpi, POLY_TERM, d, parts, _theta0(parts, d), 32, n_cr_gen=3, burnin_gen=100)
        _lib.check(ms._libh.bpm_profile(ms._handle, 1))
        ms.run_mcmc(32 * (G + 1))
        counts.append(launches_by_kind(ms))
    assert counts[0] == counts[1], counts
    k = counts[0]
    assert k["split"] == G and k["cr_reduce"] == G, k
    assert k["fused_phase"] == 0 and k["propose"] == k["likelihood"] == k["accept"] == 2 * G, k


# row = (nan flag): NaN where the data say so
NAN_TERM = r'''
__device__ double ln_like_term(const double* t, const double* row) {
  if (row[0] != 0.0) return NAN;
  return -0.5 * (t[0] * t[0] + t[1] * t[1]) * 1e-3;
}
'''


def test_nan_in_one_problem_raises():
    from bipymc_b200 import DeMcMpi
    parts = [np.zeros((m, 1)) for m in (300, 7, 1000, 40)]
    parts[2][999, 0] = 1.0
    ms = _multi(DeMcMpi, NAN_TERM, 2, parts, [-0.5, 0.0], 32, varepsilon=1e-2)
    with pytest.raises(ValueError, match="probabilities contain NaN"):
        ms.run_mcmc(32 * 4)


@pytest.mark.parametrize("ext", [".h5", ".npz"])
def test_checkpoint_resumes_bit_for_bit(tmp_path, ext):
    from bipymc_b200 import DreamMpi
    path = str(tmp_path / ("ck" + ext))
    kw = dict(n_cr_gen=3, burnin_gen=30)
    lengths = [300, 5, 4097, 1, 777]
    seeds = [5, 9, 2, 7, 1]

    def make(seed):
        parts = _poly_ragged(lengths, 3)
        return _multi(DreamMpi, POLY_TERM, 3, parts, _theta0(parts, 3), 33, seed=seed, varepsilon=1e-3, **kw)

    a = make(seeds)
    a.run_mcmc(33 * 13)
    a.save_state(path)
    a.run_mcmc(33 * 13)
    b = make(0)
    b.load_state(path)
    assert b.problem_seeds == seeds
    b.run_mcmc(33 * 13)
    np.testing.assert_array_equal(a._hist.tensor()[:, :, :3].cpu().numpy(), b._hist.tensor()[:, :, :3].cpu().numpy())
    np.testing.assert_array_equal(a._lnl.cpu().numpy(), b._lnl.cpu().numpy())
    np.testing.assert_array_equal(a.p_cr, b.p_cr)
    np.testing.assert_array_equal(a.n_accepted, b.n_accepted)
