"""Native-RNG (Philox) mode on the GPU.

(1) step parity: the device dumps the draws its counter-based stream will use
    (bpm_dump_draws); the oracle replays them on the CPU; the device's native step must
    land on the same states (1e-12 relative).
(2) posterior quality: the reference's own statistical gates (tests/test_banana.py:66-72,
    tests/test_dblgauss.py:67-69, tests/test_100dgauss.py:67-69) plus Gelman-Rubin
    R-hat < 1.01.
(3) size-independent properties at BASELINE.json's full size (10^5 chains x 100-D):
    fused == split path bit for bit, cached likelihoods == fresh evaluation, history
    rows == states, running moments == moments of the history, counters add up.
"""
import warnings

import numpy as np
import pytest

from oracle import replay as orp
from oracle import targets as otargets

pytestmark = pytest.mark.gpu
RTOL = 1e-12


def _cfg(s):
    dream = s._algo == 1
    return dict(algo="dream" if dream else "demc", del_pairs=getattr(s, "del_pairs", 1),
                n_cr=getattr(s, "n_cr", 1), gamma_scale=getattr(s, "gamma_scale", 1.0), gamma=None,
                burnin_gen=getattr(s, "burnin_gen", 0), n_cr_gen=getattr(s, "p_cr_update_gen", 0))


def _native_vs_oracle(s, oracle_lnl, gens, k0=0, run_kwargs=None):
    run_kwargs = run_kwargs or {}
    cfg = _cfg(s)
    cfg["gamma"] = run_kwargs.get("gamma")
    N = s.n_chains
    cr = orp.CrState(cfg["n_cr"]) if cfg["algo"] == "dream" else None
    if cr is not None:
        cr.p_cr, cr.delta_m, cr.n_cr_updates = s.p_cr, s.delta_m, s.n_cr_updates
    lnl = orp.scalar_batch(oracle_lnl)
    n_acc = 0
    for g in range(gens):
        k = k0 + g
        # run_mcmc sets the run parameters; make the dump see the same ones
        s.run_mcmc(N, **run_kwargs)                       # zero generations, sets params
        tr = s._dump_native_draws(k)
        pre = s._X[:, :s.dim].cpu().numpy()
        hist = s._hist.tensor()[:, :, :s.dim].cpu().numpy()
        hv = None
        if cfg["algo"] == "dream" and hist.shape[0] > cfg["n_cr_gen"]:
            # native mode keeps running (Welford) moments: a column that never moved has
            # variance exactly 0 (-> the 1e-12 floor), where np.std would return rounding noise
            hv = np.var(hist, axis=0)
            hv[np.all(hist == hist[0], axis=0)] = 0.0
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            want = orp.replay_generation(pre, tr, cfg, lnl, k, hist_var=hv, cr=cr)
        s.run_mcmc(2 * N, _k_gen0=k, **run_kwargs)         # exactly one native generation
        got = s._X[:, :s.dim].cpu().numpy()
        err = np.abs(got - want["state"]) / np.maximum(1.0, np.abs(want["state"]))
        assert err.max() <= RTOL, "generation %d: max rel err %.3e" % (k, err.max())
        assert s.n_accepted == int(want["accept"].sum())
        assert s.n_rejected == 1 + N - int(want["accept"].sum())
        n_acc += s.n_accepted
        if cr is not None:
            # The jump statistic divides by each chain's history variance.  Native mode keeps Welford moments,
            # the oracle np.var's two-pass formula: for a chain that has moved by ~1e-9 once, BOTH lose ~7
            # digits in (x - mean), differently.  1e-6 here; the strict 1e-10 gate is the RNG-replay suite,
            # whose kernels walk the stored history exactly like np.std.
            np.testing.assert_allclose(s.p_cr, cr.p_cr, rtol=1e-6)
            assert np.array_equal(s.n_cr_updates, cr.n_cr_updates)
    return n_acc


@pytest.mark.parametrize("fused", [True, False], ids=["fused", "split"])
def test_native_dream_banana_matches_oracle_replay(fused):
    from bipymc_b200 import DreamMpi, targets
    np.random.seed(1)
    s = DreamMpi(targets.Banana_2D().ln_like, [0.0, 0.0], n_chains=11, n_cr_gen=3, burnin_gen=12,
                 seed=123, fused=fused, varepsilon=0.05)
    acc = _native_vs_oracle(s, otargets.Banana2D().ln_like, gens=16)
    assert acc > 0


@pytest.mark.parametrize("fused", [True, False], ids=["fused", "split"])
def test_native_demc_bimodal_matches_oracle_replay(fused):
    from bipymc_b200 import DeMcMpi, targets
    np.random.seed(2)
    s = DeMcMpi(targets.BimodeGauss_2D().ln_like, [0.0, 0.0], n_chains=20, seed=7, fused=fused,
                varepsilon=0.01)
    _native_vs_oracle(s, otargets.BimodeGauss2D().ln_like, gens=12, run_kwargs=dict(epsilon=1e-6))


@pytest.mark.parametrize("fused", [1, 0, 3, 5], ids=["fused", "split", "fused-ws12", "fused-v3"])
@pytest.mark.parametrize("dim,n", [(7, 9), (100, 40), (33, 17), (100, 200)])
def test_native_dream_gauss_matches_oracle_replay(dim, n, fused):
    from bipymc_b200 import DreamMpi, targets
    np.random.seed(3)
    s = DreamMpi(targets.Gauss_100D(dim=dim).ln_like, np.zeros(dim), n_chains=n, n_cr_gen=2,
                 burnin_gen=1000, seed=99, fused=fused, varepsilon=0.5)
    _native_vs_oracle(s, otargets.GaussND(dim=dim).ln_like, gens=8, k0=3)


@pytest.mark.parametrize("dim,n", [(8, 20), (64, 70), (68, 70), (104, 300), (108, 130), (112, 130)])
def test_native_dream_gauss_fused_edge_dims(dim, n):
    """Dimensions at the edges of the default fused kernel: one / two / partially filled 16-byte chunks
    per lane in the write-back map (8, 64, 68), 104 with five tiles, the largest d whose tiles fit shared
    memory (108, default variant only), and the first that does not (112: the engine falls back to the
    split path).  More than one tile, last tile partial."""
    from bipymc_b200 import DreamMpi, targets
    np.random.seed(4)
    s = DreamMpi(targets.Gauss_100D(dim=dim).ln_like, np.zeros(dim), n_chains=n, n_cr_gen=2,
                 burnin_gen=1000, seed=17, fused=1, varepsilon=0.5)
    _native_vs_oracle(s, otargets.GaussND(dim=dim).ln_like, gens=6, k0=2)


def test_native_linefit_matches_oracle_replay():
    from bipymc_b200 import DreamMpi, targets
    np.random.seed(4)
    s = DreamMpi(targets.LineFit().ln_like, [-0.8, 4.5, 0.2], n_chains=12, n_cr_gen=2, burnin_gen=50,
                 seed=5, varepsilon=1e-4)
    _native_vs_oracle(s, otargets.LineFit().ln_like, gens=10)


def test_native_expfit_matches_oracle_replay():
    """5-parameter relaxation fit of examples/ex_exp_fit.py (d = 5: generic split path with the
    built-in device likelihood)."""
    from bipymc_b200 import DreamMpi, DeMcMpi, targets
    th0 = [12.0, 1.5, 0.6, 1e-3, 2e-3]
    veps = np.asarray([1e-2, 1e-2, 1e-3, 1e-8, 1e-9]) * 1e-2          # ex_exp_fit.py:135
    np.random.seed(5)
    s = DreamMpi(targets.ExpFit().ln_like, th0, n_chains=14, n_cr_gen=2, burnin_gen=1000, seed=8,
                 varepsilon=veps)
    _native_vs_oracle(s, otargets.ExpFit().ln_like, gens=10, k0=0)
    np.random.seed(6)
    s = DeMcMpi(targets.ExpFit().ln_like, th0, n_chains=9, seed=9, varepsilon=veps)
    _native_vs_oracle(s, otargets.ExpFit().ln_like, gens=6, k0=8)


def test_seed_reproducible_and_seed_sensitive():
    from bipymc_b200 import DreamMpi, targets
    outs = []
    for seed in (11, 11, 12):
        np.random.seed(0)
        s = DreamMpi(targets.Banana_2D().ln_like, [0.0, 0.0], n_chains=64, seed=seed)
        s.run_mcmc(64 * 40)
        outs.append(s._hist.tensor().cpu().numpy())
    assert np.array_equal(outs[0], outs[1])
    assert not np.array_equal(outs[0], outs[2])


# ---------------------------------------------------------------- posterior gates
def test_banana_posterior_gates_like_reference_test():
    """tests/test_banana.py:43-44,66-72: fraction of post-burn-in samples inside the
    pdf > 0.18 / pdf > 0.018 regions within 0.05 of the truth, DE-MC 20 / DREAM 10 chains."""
    from bipymc_b200 import DeMcMpi, DreamMpi, targets
    banana = targets.Banana_2D(sigma1=1.0, sigma2=1.0)
    np.random.seed(42)
    y1, y2 = banana.rvs(1000000)
    f50 = np.count_nonzero(banana.check_prob_lvl(y1, y2, 0.18)) / y1.size
    f95 = np.count_nonzero(banana.check_prob_lvl(y1, y2, 0.018)) / y1.size
    n_samples, n_burn = 100000, 20000
    for s in (DeMcMpi(banana.ln_like, [0.0, 0.0], n_chains=20, seed=1),
              DreamMpi(banana.ln_like, [0.0, 0.0], n_chains=10, n_cr_gen=50, burnin_gen=2000, seed=2)):
        s.run_mcmc(n_samples)
        theta, sig, chain = s.param_est(n_burn=n_burn)
        assert chain.shape == (n_samples - n_burn, 2)
        g50 = np.count_nonzero(banana.check_prob_lvl(chain[:, 0], chain[:, 1], 0.18)) / chain.shape[0]
        g95 = np.count_nonzero(banana.check_prob_lvl(chain[:, 0], chain[:, 1], 0.018)) / chain.shape[0]
        assert abs(g50 - f50) < 0.05 and abs(g95 - f95) < 0.05
        assert 0.1 < s.acceptance_fraction < 0.6


def test_bimodal_posterior_mean_like_reference_test():
    """tests/test_dblgauss.py:43-44,67-69: mean = (1.5, 1.5) +- 0.1."""
    from bipymc_b200 import DeMcMpi, DreamMpi, targets
    tgt = targets.BimodeGauss_2D()
    for s in (DeMcMpi(tgt.ln_like, [0.0, 0.0], n_chains=20, seed=3),
              DreamMpi(tgt.ln_like, [0.0, 0.0], n_chains=10, n_cr_gen=50, burnin_gen=2000, seed=4)):
        s.run_mcmc(100000)
        theta, sig, chain = s.param_est(n_burn=40000)
        assert abs(theta[0] - 1.5) < 0.1 and abs(theta[1] - 1.5) < 0.1


def test_large_population_posterior_and_rhat():
    """Wide population, long run: mean / covariance of the banana's underlying Gaussian
    coordinates within Monte-Carlo error and Gelman-Rubin R-hat < 1.01 over the second
    half of the chains (north_star's convergence gate)."""
    from bipymc_b200 import DreamMpi, targets
    from bipymc_b200.diagnostics import gelman_rubin
    banana = targets.Banana_2D()
    np.random.seed(0)
    N, G = 1024, 20000
    s = DreamMpi(banana.ln_like, [0.0, 0.0], n_chains=N, seed=21, burnin_gen=2000, n_cr_gen=50,
                 varepsilon=1.0)
    s.run_mcmc(N * (G + 1))
    h = s._hist.tensor()[G // 2:, :, :2]
    rhat = gelman_rubin(h)
    print("banana R-hat", rhat, "acc", s.acceptance_fraction, "p_cr", s.p_cr)
    assert np.all(rhat < 1.01), rhat
    flat = h.reshape(-1, 2).cpu().numpy()
    x1, x2 = banana.inv_transform(flat[:, 0], flat[:, 1])
    # underlying N(0, [[1, .9], [.9, 1]])
    assert abs(x1.mean()) < 0.02 and abs(x2.mean()) < 0.02, (x1.mean(), x2.mean())
    c = np.cov(np.stack([x1[::7], x2[::7]]))
    assert abs(c[0, 0] - 1.0) < 0.03 and abs(c[1, 1] - 1.0) < 0.03 and abs(c[0, 1] - 0.9) < 0.03, c


def test_gauss100_posterior_like_reference_test():
    """tests/test_100dgauss.py:67-69 (mean[0], mean[1] = 0 +- 0.2), plus every marginal
    mean / variance (var_i = i + 1, d100_gauss.py:16) and Gelman-Rubin R-hat < 1.01.
    100-D DREAM has an autocorrelation time of several hundred generations, so the gate
    needs ~10^5 generations; history is off and everything comes from the running
    per-chain moments (reset after burn-in)."""
    from bipymc_b200 import DreamMpi, targets
    tgt = targets.Gauss_100D()
    np.random.seed(0)
    N, G_burn, G = 512, 20000, 80000
    s = DreamMpi(tgt.ln_like, np.zeros(100), n_chains=N, seed=5, burnin_gen=2000, n_cr_gen=50,
                 varepsilon=2.0 * (np.arange(100) + 1.0), history="none")
    s.run_mcmc(N * (G_burn + 1))
    s.reset_moments()
    s.track_covariance(True)
    s.run_mcmc(N * (G + 1), _k_gen0=G_burn)
    assert s._mom_len == G + 1
    rhat = s.rhat()
    mean, sd = s.moment_estimates()
    var = sd ** 2
    truth = np.arange(100) + 1.0
    print("gauss100 max R-hat %.4f acc %.3f max|mean|/sd %.3f var ratio [%.3f, %.3f] p_cr %s" % (
        rhat.max(), s.acceptance_fraction, np.max(np.abs(mean) / np.sqrt(truth)),
        (var / truth).min(), (var / truth).max(), s.p_cr))
    assert abs(mean[0]) < 0.2 and abs(mean[1]) < 0.2
    assert np.all(np.abs(mean) < 0.05 * np.sqrt(truth))
    np.testing.assert_allclose(var, truth, rtol=0.05)
    assert np.all(rhat < 1.01), rhat.max()
    assert 0.05 < s.acceptance_fraction < 0.7
    # the full posterior covariance, off-diagonals included: Sigma_ij = rho sqrt(i+1) sqrt(j+1), rho = 0.5
    # (d100_gauss.py:14-22), from the device cross-moment accumulator.  Monte-Carlo standard error of a
    # correlation at n_eff ~ N G / tau ~ 512 * 8e4 / 5e2 ~ 8e4 is (1 - rho^2) / sqrt(n_eff) ~ 0.003; the
    # maximum over 4 950 pairs sits near 4 sigma.
    cm, cov = s.covariance_estimate()
    np.testing.assert_allclose(cm, mean, rtol=0, atol=0.05)       # same chains, one generation apart
    sdv = np.sqrt(np.diag(cov))
    corr = cov / np.outer(sdv, sdv)
    off = corr[~np.eye(100, dtype=bool)]
    print("gauss100 off-diagonal correlation: mean %.4f min %.4f max %.4f (truth 0.5)" % (off.mean(), off.min(), off.max()))
    assert abs(off.mean() - 0.5) < 0.005
    assert np.all(np.abs(off - 0.5) < 0.03), (off.min(), off.max())
    np.testing.assert_allclose(np.diag(cov), truth, rtol=0.05)
    ref_cov = tgt.cov
    assert np.max(np.abs(cov - ref_cov) / np.sqrt(np.outer(truth, truth))) < 0.05


def test_streaming_rhat_and_moments_match_history():
    """rhat() / moment_estimates() from running moments == the same statistics computed
    from the stored history (bipymc_b200.diagnostics.gelman_rubin, param_est)."""
    from bipymc_b200 import DreamMpi, targets
    from bipymc_b200.diagnostics import gelman_rubin
    np.random.seed(1)
    s = DreamMpi(targets.Banana_2D().ln_like, [0.0, 0.0], n_chains=64, seed=3, varepsilon=0.5)
    s.run_mcmc(64 * 401)
    h = s._hist.tensor()[:, :, :2]
    np.testing.assert_allclose(s.rhat(), gelman_rubin(h), rtol=1e-9)
    m, sd, _ = s.param_est(0)
    gm, gsd = s.moment_estimates()
    np.testing.assert_allclose(gm, m, rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(gsd, sd, rtol=1e-9)


# ---------------------------------------------------------------- full-size properties
def test_full_size_properties_1e5_chains_100d():
    import torch
    from bipymc_b200 import DreamMpi, targets
    tgt = targets.Gauss_100D()
    N, d, G = 100000, 100, 6
    runs = []
    for fused in (1, 0, 3, 5):     # 1 = TMA-staged gathers (v4, default), 3 = 12 producers, 5 = register gathers (v3)
        np.random.seed(0)
        s = DreamMpi(tgt.ln_like, np.zeros(d), n_chains=N, seed=77, burnin_gen=1000, n_cr_gen=2,
                     fused=fused, varepsilon=1.0)
        s.run_mcmc(N * (G + 1))
        runs.append(s)
    a, b, c3, c5 = runs
    ha, hb = a._hist.tensor(), b._hist.tensor()
    assert ha.shape == (G + 1, N, d)
    # v3 and v4 differ only in HOW the partner rows reach the proposal stage: identical bits everywhere
    assert torch.equal(ha, c5._hist.tensor()) and torch.equal(a._lnl, c5._lnl)
    assert torch.equal(a._mean, c5._mean) and torch.equal(a._m2, c5._m2)
    del c5
    # every variant builds identical proposals and makes identical accept decisions; the
    # default variant sums the quadratic form in DMMA fragment order, so its cached
    # likelihoods agree with the scalar variants to rounding, theirs among themselves exactly
    assert torch.equal(ha, hb), "fused and split paths must produce the same chains"
    assert torch.equal(hb, c3._hist.tensor())
    assert torch.equal(b._lnl, c3._lnl)
    assert torch.allclose(a._lnl, b._lnl, rtol=1e-13, atol=0.0)
    del c3
    np.testing.assert_allclose(a.p_cr, b.p_cr, rtol=1e-12)
    # history row G == live population; every chain moved at most once per generation
    assert torch.equal(ha[G], a._X)
    # cached likelihood == fresh evaluation of the current state
    fresh = a._eval_lnl_rows(a._X)
    assert torch.equal(fresh, b._lnl) and torch.allclose(fresh, a._lnl, rtol=1e-13, atol=0.0)
    # counters add up: every chain stepped once per generation
    assert a.n_accepted + a.n_rejected == N * G + 1
    changed = int((ha[1:] != ha[:-1]).any(dim=2).sum().item())
    assert changed == a.n_accepted
    # running moments == moments of the stored history
    mean = ha.mean(dim=0)
    m2 = ((ha - mean[None]) ** 2).sum(dim=0)
    assert torch.allclose(a._mean, mean, rtol=1e-12, atol=1e-13)
    assert torch.allclose(a._m2, m2, rtol=1e-10, atol=1e-12)
    # the a/b split: within a generation a chain's partners come from the other half, so a
    # rejected chain is bit-identical to its previous row (no partial writes)
    same = (ha[1:] == ha[:-1]).all(dim=2)
    assert int(same.sum().item()) == N * G - a.n_accepted


# ---------------------------------------------------------------- the other BASELINE configs
def test_config5_shape_1000d_gauss_matches_oracle_replay():
    """configs[4] at a size the oracle finishes: DREAM on the 1000-D correlated Gaussian with
    the direct log-density (the reference's log(pdf) underflows there, SURVEY.md section 0);
    generic split path (d > 112), native Philox draws replayed by the oracle."""
    from bipymc_b200 import DreamMpi, targets
    np.random.seed(11)
    dim, n = 1000, 12
    tgt = targets.Gauss_100D(dim=dim)
    assert tgt.log_of_pdf is False
    s = DreamMpi(tgt.ln_like, np.zeros(dim), n_chains=n, n_cr_gen=2, burnin_gen=1000, seed=5, varepsilon=0.5)
    _native_vs_oracle(s, otargets.GaussND(dim=dim, use_logpdf=True).ln_like, gens=4, k0=4)


def test_config3_bimodal_1e6_chains_outlier_reset_and_cr_adaptation():
    """configs[2] at full size: DREAM on the bimodal Gaussian with 10^6 chains, CR adaptation
    and the IQR outlier reset ON.  Size-independent properties: counters add up, cached
    likelihoods equal a fresh evaluation, p_cr is a distribution that moved off uniform, the
    population mean reaches the reference's gate (tests/test_dblgauss.py:67-69) and the two modes carry their
    weights (0.25 / 0.75)."""
    import torch
    from bipymc_b200 import DreamMpi, targets
    tgt = targets.BimodeGauss_2D(log_of_pdf=False)      # log-sum-exp: finite in the far tails
    N = 1000000
    np.random.seed(1)
    s = DreamMpi(tgt.ln_like, [0.0, 0.0], n_chains=N, seed=17, varepsilon=1.0, history="none",
                 burnin_gen=150, n_cr_gen=20, outlier_gen=50)
    G1 = 150
    s.run_mcmc(N * (G1 + 1))
    assert s.n_accepted + s.n_rejected == N * G1 + 1
    p = s.p_cr
    assert abs(p.sum() - 1.0) < 1e-12 and np.all(p > 0) and np.abs(p - 1.0 / 3).max() > 1e-3
    assert np.all(s.n_cr_updates > 0)
    assert s.last_outlier_stats["threshold"] < s.last_outlier_stats["q1"]
    s.reset_moments()
    G2 = 200
    s.run_mcmc(N * (G2 + 1), _k_gen0=G1)
    fresh = s._eval_lnl_rows(s._X)
    assert torch.equal(fresh, s._lnl)
    mean, std = s.moment_estimates()
    assert abs(mean[0] - 1.5) < 0.1 and abs(mean[1] - 1.5) < 0.1, mean
    # each chain saw only 200 post-burn-in rows of a bimodal target: the per-chain means
    # differ (chains sit in one mode), so R-hat is a mixing statement, not < 1.01 here;
    # the population statistic that must hold is the mode weight (0.25 / 0.75)
    frac_hi = float((s._X[:, 0] + s._X[:, 1] > 2.0).double().mean().item())
    assert abs(frac_hi - 0.75) < 0.03, frac_hi
    assert 0.05 < s.acceptance_fraction < 0.7


def test_checkpoint_roundtrip_resumes_the_same_chains(tmp_path):
    """save_state / load_state / warm_start (demc.py:198-233, demc.py:46-51): chains restored
    bit for bit, and -- the extension over the reference -- the Philox seed and CR adaptation
    state travel with them, so a resumed run continues exactly like an uninterrupted one."""
    from bipymc_b200 import DreamMpi, targets
    tgt = targets.Banana_2D()
    f = str(tmp_path / "ckpt.h5")
    kw = dict(n_chains=24, n_cr_gen=3, burnin_gen=1000, varepsilon=0.3)
    np.random.seed(4)
    a = DreamMpi(tgt.ln_like, [0.0, 0.0], seed=31, **kw)
    a.run_mcmc(24 * 11)
    a.save_state(f)
    # the file IS the reference's HDF5 layout (chain.py:59-93): /chains/chain_id_<id>, gzip, (T, dim) float64 --
    # written by h5py where it imports, by bipymc_b200.h5lite (same on-disk format) where it does not
    from bipymc_b200 import h5lite
    assert open(f, "rb").read(8) == b"\x89HDF\r\n\x1a\n"
    with h5lite.File(f, "r") as h5f:
        assert h5f["/chains"].keys() == sorted("chain_id_%d" % i for i in range(24))
        for i in (0, 7, 23):
            ds = h5f["/chains/chain_id_%d" % i]
            assert ds.shape == (11, 2) and ds.dtype == np.float64 and ds.compression == "gzip"
            np.testing.assert_array_equal(ds[:], a.am_chains[i].chain)
        assert int(h5f["/chains"].attrs["b200_seed"]) == 31
    a.run_mcmc(24 * 6)
    np.random.seed(99)
    b = DreamMpi(tgt.ln_like, [0.0, 0.0], warm_start=True, h5_file=f, **kw)      # no seed given
    assert b._seed == 31
    assert b.am_chains[3].chain_len == 11
    np.testing.assert_array_equal(b.am_chains[3].chain, a.am_chains[3].chain[:11])
    b.run_mcmc(24 * 6)
    np.testing.assert_array_equal(b.super_chain, a.super_chain)
    np.testing.assert_allclose(b.p_cr, a.p_cr, rtol=1e-13)
    assert np.array_equal(b.n_cr_updates, a.n_cr_updates)
    # ragged / foreign files are rejected like the reference does (bare RuntimeError, demc.py:232)
    c = DreamMpi(tgt.ln_like, [0.0, 0.0], seed=1, n_chains=25)
    with pytest.raises(RuntimeError):
        c.load_state(f)


@pytest.mark.parametrize("dim,n,shift", [(128, 300, False), (200, 1000, True), (1000, 777, False), (1000, 64, True),
                                         (114, 50, True)])
def test_large_d_quadratic_form_matches_numpy(dim, n, shift):
    """bpm_eval_lnl for d > 112 (FP64 tensor-pipe GEMM kernel, gauss_dmma.cuh): values agree with
    the host's scipy-style evaluation to 1e-12 relative, including a non-zero mean, ragged n and
    column / k tails that are not multiples of the tile."""
    import torch
    from bipymc_b200 import DreamMpi, targets
    rs = np.random.RandomState(dim + n)
    mean = rs.randn(dim) if shift else None
    t = targets.Gauss_100D(dim=dim, mean=mean, log_of_pdf=False)
    np.random.seed(0)
    s = DreamMpi(t.ln_like, np.zeros(dim), n_chains=8, seed=1, varepsilon=1.0)
    X = rs.randn(n, dim) * np.sqrt(np.arange(dim) + 1.0)
    rows = torch.zeros((n, s._ld), dtype=torch.float64, device=s._device)
    rows[:, :dim] = torch.from_numpy(X).to(s._device)
    got = s._eval_lnl_rows(rows).cpu().numpy()
    want = np.array([t.ln_like(x) for x in X])
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-10)


@pytest.mark.parametrize("adapt", [False, True], ids=["noadapt", "adapt"])
@pytest.mark.parametrize("pinned", [True, False])
def test_host_buffer_entry_equals_device_resident_generations(pinned, adapt):
    """bpm_generations_host (the end-to-end entry: HOST population in, HOST population out) must
    leave exactly the population a device-resident run produces -- both with pinned buffers (only
    the rows that moved are written back by the device) and with pageable ones (full copy) -- and,
    with crossover adaptation on, the same p_cr: the entry keeps the chains' running moments on the
    device between calls (dream.py:119-140 needs np.std of every chain's history)."""
    import ctypes as C
    import torch
    from bipymc_b200 import DreamMpi, targets, _lib
    N, d, G = 4096, 100, 7
    tgt = targets.Gauss_100D()
    kw = dict(burnin_gen=1000, n_cr_gen=2) if adapt else dict(burnin_gen=0)
    np.random.seed(1)
    a = DreamMpi(tgt.ln_like, np.zeros(d), n_chains=N, seed=8, varepsilon=1.0, history="none", **kw)
    np.random.seed(1)
    b = DreamMpi(tgt.ln_like, np.zeros(d), n_chains=N, seed=8, varepsilon=1.0, history="none", **kw)
    b.run_mcmc(N)                                   # sets run parameters, evaluates the initial likelihoods
    Xh = torch.empty((N, b._ld), dtype=torch.float64)
    Lh = torch.empty((N,), dtype=torch.float64)
    if pinned:
        Xh, Lh = Xh.pin_memory(), Lh.pin_memory()
    Xh.copy_(b._X.cpu()); Lh.copy_(b._lnl.cpu())
    moved = 0
    for g in range(G):
        before = Xh.clone()
        _lib.check(b._libh.bpm_generations_host(b._handle, Xh.data_ptr(), Lh.data_ptr(), g, 1 + g, 1))
        nb = C.c_uint64()
        _lib.check(b._libh.bpm_last_d2h_bytes(b._handle, C.byref(nb)))
        rows = int((before != Xh).any(dim=1).sum())
        moved += rows
        if pinned:       # accepted rows stored from inside the kernels + one copy of the cached likelihoods
            assert nb.value == rows * b._ld * 8 + N * 8 + 16
        else:
            assert nb.value == N * (b._ld + 1) * 8
    a.run_mcmc(N * (G + 1))
    assert torch.equal(a._X.cpu(), Xh) and torch.equal(a._lnl.cpu(), Lh)
    assert moved == a.n_accepted
    if adapt:
        assert a.n_cr_updates.sum() > 0
        assert np.array_equal(a.p_cr, b.p_cr) and np.array_equal(a.delta_m, b.delta_m)
